/*
 * rrtk.h -- C ABI of librrtk.so: the B200 (sm_100a) tree-expansion hot path of rrtplanner.
 *
 * The reference (rland93/rrtplanner) has no FFI layer: its hot path is a set of Python methods on
 * the planner classes of rrtplanner/rrt.py.  Each entry point below names the reference interface it
 * replaces (file:line in /root/reference).  The Python classes in rrtplanner_b200/rrt.py bind these
 * symbols with ctypes (see INTEGRATION.md for the stub a reference maintainer would add).
 *
 * Conventions
 *   - plain C types only; every pointer is caller-owned.  "d_" parameters are DEVICE pointers,
 *     "h_" parameters are HOST pointers (pinned memory makes the copies asynchronous).
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream).  Device-pointer entry
 *     points only enqueue work on it; host-pointer entry points synchronise it before returning.
 *   - every function returns RRTK_OK (0) or a negative rrtk_status; rrtk_last_error() gives text.
 *   - occupancy grids are (W, H) arrays indexed og[x*H + y] exactly like the reference's og[x, y]
 *     (rrt.py:218); any non-zero cell is an obstacle (rrt.py:191).
 *   - coordinates are int32 in the ABI; the planner kernels require 0 <= x < W <= 16384,
 *     0 <= y < H <= 16384 and n <= 65534.
 *
 * Bit grid layout ("tiled"): the grid is cut into 32x32-cell tiles, tile (tx, ty) = (x>>5, y>>5),
 * tiles stored row-major over (tx, ty) with TY = ceil(H/32) tiles per row; one tile is 32
 * consecutive uint32 words (128 bytes, one L2 line); word (x & 31) of a tile holds the 32 cells
 * y = 32*ty .. 32*ty+31 of row x, bit (y & 31).  Cells outside (W, H) are set (obstacle).
 */
#ifndef RRTK_H
#define RRTK_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RRTK_VERSION 100

typedef enum {
    RRTK_OK = 0,
    RRTK_ERR_INVALID = -1,   /* bad argument (NULL pointer, size out of range, point outside grid) */
    RRTK_ERR_CAPACITY = -2,  /* problem does not fit the kernel's shared-memory / index limits */
    RRTK_ERR_CUDA = -3,      /* a CUDA runtime call failed; see rrtk_last_error() */
    RRTK_ERR_NODEVICE = -4   /* no CUDA device visible */
} rrtk_status;

typedef enum {
    RRTK_STANDARD = 0,       /* RRTStandard.plan      rrt.py:386-447 */
    RRTK_STAR = 1,           /* RRTStar.plan          rrt.py:466-556 */
    RRTK_INFORMED = 2        /* RRTStarInformed.plan  rrt.py:653-758 */
} rrtk_kind;

/* one plan = one (world, start, goal) triple; 64 bytes */
typedef struct {
    int32_t world;           /* index of the bit grid this plan runs on */
    int32_t start_x, start_y;
    int32_t goal_x, goal_y;
    int32_t reserved[3];
    double rot[4];           /* row-major 2x2 of rotation_to_world_frame (rrt.py:601-613); informed only */
} rrtk_plan_desc;

/* per-plan statistics, int64 slots (rrtk_plan_batch writes RRTK_STAT_COUNT of them per plan) */
enum {
    RRTK_STAT_J = 0,           /* filled vertices before goal connection (the reference's j) */
    RRTK_STAT_VGOAL,           /* goal vertex id: j when connected, else 0 (rrt.py:319,330-331) */
    RRTK_STAT_FOUND,           /* 1 when the goal row was appended */
    RRTK_STAT_CHECKS,          /* collision checks executed on the device (parallel form) */
    RRTK_STAT_CELLS,           /* grid cells those checks tested (first hit inclusive) */
    RRTK_STAT_FIRST_SOL_ITER,  /* informed: iteration of the first solution vertex, else -1 */
    RRTK_STAT_ELL_ITERS,       /* informed: iterations sampled from the ellipse */
    RRTK_STAT_NN_PAIRS,        /* sum over iterations of filled vertices scanned */
    RRTK_STAT_RING_MEMBERS,    /* sum over accepted iterations of |within(r_rewire)| */
    RRTK_STAT_ACCEPTED,        /* accepted samples */
    RRTK_STAT_RESERVED0,
    RRTK_STAT_RESERVED1,
    RRTK_STAT_COUNT
};

int rrtk_version(void);
const char *rrtk_last_error(void);
/* number of visible CUDA devices (0 if none; never fails) */
int rrtk_device_count(void);
int rrtk_set_device(int device);
/* SM count and opt-in shared memory per block of the current device */
int rrtk_device_info(int *sm_count, int *smem_optin_bytes);

/* Roofline denominators measured on the device at hand (bench.py; SURVEY.md section 8(d) bounds the nearest / radius
 * scan of rrt.py:131-181 by shared-memory bandwidth and the collision walk of rrt.py:183-229 by L2 bandwidth, and
 * MEASURED_PEAKS.json holds neither).  Each call launches one read sweep on `stream` and reports the bytes it reads;
 * the caller times it with events.  rrtk_peak_l2_read: `passes` sweeps over d_buf (choose `bytes` between the L1 and
 * the L2 size; warm L2 with one untimed call).  rrtk_peak_smem_read: one block per SM reads its shared memory `iters`
 * times with conflict-free 16-byte loads (smem_bytes <= 0: as much as a block may have). */
int rrtk_peak_l2_read(const void *d_buf, size_t bytes, int passes, uint32_t *d_sink, int64_t *bytes_read, void *stream);
int rrtk_peak_smem_read(int smem_bytes, int iters, uint32_t *d_sink, int64_t *bytes_read, void *stream);

/* ---- occupancy grids ------------------------------------------------------------------------- */
/* uint32 words of one tiled bit grid */
size_t rrtk_grid_words(int W, int H);

/* K0.  Replaces the `og[x, y] != 0` test of rrt.py:218 by a packed copy: d_og is nworlds
 * consecutive (W,H) uint8 grids, d_bits receives nworlds * rrtk_grid_words(W,H) words. */
int rrtk_pack_grid(const uint8_t *d_og, int nworlds, int W, int H, uint32_t *d_bits, void *stream);

/* inverse of rrtk_pack_grid: d_og receives nworlds (W,H) uint8 grids of 0 / 1 */
int rrtk_unpack_grid(const uint32_t *d_bits, int nworlds, int W, int H, uint8_t *d_og, void *stream);

/* free-space index for RRT.sample_all_free (rrt.py:64,231-240): d_rowcum[w*(W+1) + x] = number of
 * free cells in rows < x of world w (so entry W is nfree, the size of the reference's `free`). */
int rrtk_free_rows(const uint32_t *d_bits, int nworlds, int W, int H, int32_t *d_rowcum, void *stream);

/* Synthetic worlds (measurement fixture; oggen.py:7-45 semantics, integer value-noise fBm that is
 * bit-identical to rrtplanner_b200/worlds.py).  World i uses seed seeds[i].  d_scratch must hold
 * nworlds * W * H int32 + 2 * nworlds int32. */
int rrtk_gen_worlds(const int32_t *d_seeds, int nworlds, int W, int H, int thresh_permille,
                    int32_t *d_scratch, uint8_t *d_og, void *stream);

/* Obstacle inflation of the replanning caller (anim.py:79-87, the frame loop that calls set_og + plan):
 *   dilated = scipy.ndimage.binary_dilation(og, iterations)   -- 4-connected cross, outside = free
 *   out     = og | (dilated & ~og & ~hole)                     -- hole = clamped square the agent stands in
 * Output grid o (o < nout, nout >= nworlds) is made from source world o % nworlds, so many agents can share one
 * dilation of one frame.  d_holes: per OUTPUT grid (px, py, size) int32: cells [px, px+size) x [py, py+size),
 * clipped to the grid, keep no buffer (anim.py:82-86 uses size = 2 * iterations); NULL or size 0 = no hole.
 * d_out holds nout grids, d_scratch 2 * nworlds grids (rrtk_grid_words(W,H) words each); neither may alias
 * d_bits.  iterations >= 0 (0 = no buffer). */
int rrtk_inflate_grid(const uint32_t *d_bits, int nworlds, int W, int H, int iterations, const int32_t *d_holes,
                      int nout, uint32_t *d_out, uint32_t *d_scratch, void *stream);

/* ---- K1: RRT.collisionfree (rrt.py:183-229), batched ------------------------------------------- */
/* d_segs: nseg x (ax, ay, bx, by) int32, all points inside the grid.  d_world: optional per-segment
 * world index (NULL = world 0).  d_free[s] = 1 iff the walk a->b meets no obstacle (both ends
 * included).  d_cells[s] (optional) = number of cells the reference's loop reads before returning
 * (index of first obstacle + 1, or max(|dx|,|dy|) + 1). */
int rrtk_collision_segments(const uint32_t *d_bits, int W, int H, const int32_t *d_segs,
                            const int32_t *d_world, int64_t nseg, uint8_t *d_free, int32_t *d_cells,
                            void *stream);

/* ---- K1b: the same function on a clearance field ------------------------------------------------- */
/* d_clear[w*W*H + x*H + y] = min(cap, Chebyshev distance of cell (x, y) of world w to the nearest obstacle
 * cell or to the outside of the grid); 0 on obstacles.  2 <= cap <= 255.  d_scratch: 2 * nworlds *
 * rrtk_grid_words(W,H) words.  Built once per grid (cap - 1 dilation passes). */
int rrtk_clearance_field(const uint32_t *d_bits, int nworlds, int W, int H, int cap, uint8_t *d_clear,
                         uint32_t *d_scratch, void *stream);
/* rrtk_collision_segments with identical outputs (verdict and cells the reference's loop reads), walking the
 * clearance field: a cell with clearance d proves the next d - 1 cells of the walk free (rrt.py:183-229 moves
 * at most one cell per axis per step), so long free stretches cost one read.  One thread per segment. */
int rrtk_collision_segments_cf(const uint8_t *d_clear, int W, int H, const int32_t *d_segs, const int32_t *d_world,
                               int64_t nseg, uint8_t *d_free, int32_t *d_cells, void *stream);

/* Directional form of the same idea: eight fields per world, one per octant of a walk (which axis is the major one,
 * sign of dx, sign of dy -- rrt.py:199-215 fixes all three for a segment).  The field of octant o holds, per cell, the
 * depth (capped) of the obstacle-free cone the walk can reach from that cell, so obstacles beside or behind the walk do
 * not shorten the step: about half the reads of the isotropic field on cfg2, at 8 bytes per cell.
 *   o = 4 * (|dx| >= |dy|) + 2 * (dx > 0) + (dy > 0);   d_clear8[((w * 8 + o) * W + x) * H + y],  2 <= cap <= 255. */
int rrtk_clearance_field_dir(const uint32_t *d_bits, int nworlds, int W, int H, int cap, uint8_t *d_clear8, void *stream);
/* rrtk_collision_segments with identical outputs, walking the directional fields of rrtk_clearance_field_dir. */
int rrtk_collision_segments_cfd(const uint8_t *d_clear8, int W, int H, const int32_t *d_segs, const int32_t *d_world,
                                int64_t nseg, uint8_t *d_free, int32_t *d_cells, void *stream);

/* The same with every octant split at slope 1/2 (sixteen fields per world, 16 bytes per cell): a walk whose minor / major
 * ratio is at most 1/2 strays at most ceil(i / 2) cells sideways in i steps, a steeper one at least floor(i / 2), so each half
 * has a narrower free cone and the walk takes longer steps again (cfg2: 3.9 reads per segment instead of 4.9).
 *   field index = 2 * o + (2 * min(|dx|, |dy|) > max(|dx|, |dy|)),  o as above;   d_clear16[((w * 16 + f) * W + x) * H + y]. */
int rrtk_clearance_field_dir16(const uint32_t *d_bits, int nworlds, int W, int H, int cap, uint8_t *d_clear16, void *stream);
int rrtk_collision_segments_cfd16(const uint8_t *d_clear16, int W, int H, const int32_t *d_segs, const int32_t *d_world,
                                  int64_t nseg, uint8_t *d_free, int32_t *d_cells, void *stream);

/* ---- K2: RRT.near(points, x)[0] (rrt.py:131-155), batched, pinned tie rule (lowest index) ------- */
/* d_pts: npts x (x, y) int32.  d_queries: nq x (x, y).  d_count (optional): query q only sees the
 * first d_count[q] points (the filled prefix of the tree); NULL = all npts.  d_idx[q] = nearest
 * vertex, d_d2[q] (optional) = its exact squared distance. */
int rrtk_nearest_batch(const int32_t *d_pts, int npts, const int32_t *d_queries, const int32_t *d_count,
                       int nq, int32_t *d_idx, int64_t *d_d2, void *stream);

/* same for floating-point vertices / queries (numpy semantics: key = sqrt(dx*dx + dy*dy) in IEEE
 * double, no contraction); d_dist[q] (optional) = that key */
int rrtk_nearest_batch_f64(const double *d_pts, int npts, const double *d_queries, const int32_t *d_count,
                           int nq, int32_t *d_idx, double *d_dist, void *stream);

/* ---- K3: RRT.within(points, x, r) (rrt.py:157-181), batched --------------------------------------- */
/* d_out[q*cap .. ] receives the ascending indices with d^2 < r*r (strict), d_len[q] their number
 * (may exceed cap: only the first cap are stored). */
int rrtk_within_batch(const int32_t *d_pts, int npts, const int32_t *d_queries, const int32_t *d_count,
                      int nq, double r, int cap, int32_t *d_out, int32_t *d_len, void *stream);

/* floating-point form: dx*dx + dy*dy < r*r in IEEE double -- the reference's own known-answer test
 * calls within() with x = [0.5, 0.5] (tests/test_rrt.py:116-119) */
int rrtk_within_batch_f64(const double *d_pts, int npts, const double *d_queries, const int32_t *d_count,
                          int nq, double r, int cap, int32_t *d_out, int32_t *d_len, void *stream);

/* distance keys for the full ordering RRT.near returns (rrt.py:150-155): d_d2[i] = |pts[i]-q|^2 */
int rrtk_dist2(const int32_t *d_pts, int npts, int qx, int qy, int64_t *d_d2, void *stream);
int rrtk_dist_f64(const double *d_pts, int npts, double qx, double qy, double *d_dist, void *stream);
/* ascending stable ordering of int64 keys (ties: lowest index first) -- the pinned np.argsort */
int rrtk_argsort_i64(const int64_t *d_keys, int n, int32_t *d_perm, void *d_scratch, size_t scratch_bytes,
                     void *stream);
size_t rrtk_argsort_scratch_bytes(int n);

/* ---- sample streams: RRT.sample_all_free with numpy's PCG64 (rrt.py:85,231-240) ------------------- */
/* h_state: per plan 4 x uint64 = PCG64 {state_hi, state_lo, inc_hi, inc_lo} as numpy's
 * default_rng(seed).bit_generator.state reports them.  Writes n samples (x, y) int16 per plan:
 * sample i = free[integers(0, nfree)] of that plan's world. */
int rrtk_sample_streams(const uint32_t *d_bits, const int32_t *d_rowcum, int W, int H,
                        const rrtk_plan_desc *d_plans, int nplans, const uint64_t *d_state, int n,
                        int16_t *d_samples, void *stream);

/* Same, for a planner object that is used again (the replanning caller, anim.py:92-93: one rand_gen per
 * object, rrt.py:85, keeps running across plan() calls): d_state is updated in place to the generator
 * state after the n draws, d_carry (2 x uint32 per plan: numpy's has_uint32, uinteger; zero for a fresh
 * generator) likewise. */
int rrtk_sample_streams_carry(const uint32_t *d_bits, const int32_t *d_rowcum, int W, int H,
                              const rrtk_plan_desc *d_plans, int nplans, uint64_t *d_state, uint32_t *d_carry,
                              int n, int16_t *d_samples, void *stream);

/* The unit-disc stream of the ellipse phase of RRTStarInformed.plan (rrt.py:240, 579-587, 694-701), from the same
 * generator: the reference draws free[choice(nfree)] in iterations 0 .. f (f = the first solution iteration) and then
 * unitball() = two uniform(0, 1) draws per iteration.  Per plan p (world d_plans[p].world, nfree = d_rowcum[world*(W+1)+W]):
 *   d_state    PCG64 start state as for rrtk_sample_streams; d_carry (optional, NULL = zero) has_uint32 / uinteger
 *   d_first    f = d_first[p * first_stride] (int64; -1 = no solution): the probe's statistics work directly, e.g. K7 stats
 *              + RRTK_STAT_FIRST_SOL_ITER or K8 stats + RRTK_STAT2_FIRST_SOL with stride RRTK_STAT_COUNT
 *   d_balls    nplans x n x 2 doubles: row i > f = (sqrt(u1) cos(2 pi u2), sqrt(u1) sin(2 pi u2)) of the i-th iteration's two
 *              uniforms after the min(f + 1, n) bounded draws; rows <= f and every row when f < 0 are 0.0.  The uniforms,
 *              sqrt and products are bit-exact, cos / sin are the device's (<= 2 ulp from numpy's)
 *   d_state_out, d_carry_out (optional) the generator as the planner object holds it after plan(), for a next plan():
 *              state after the bounded draws and 2 * (n - 1 - f) 64-bit outputs, carry as the bounded draws left it.
 *              May alias d_state / d_carry.
 * This replaces the host side of RRTStarInformed.plan (rrtplanner_b200/rrt.py: generator advance + unitball() loop), so
 * a probe launch (d_balls == NULL in rrtk_plan_batch), this call and the full launch reproduce a seeded planner object. */
int rrtk_ball_streams(const int32_t *d_rowcum, int W, const rrtk_plan_desc *d_plans, int nplans, int n,
                      const uint64_t *d_state, const uint32_t *d_carry, const int64_t *d_first, int first_stride,
                      double *d_balls, uint64_t *d_state_out, uint32_t *d_carry_out, void *stream);

/* ---- K7: the plan() loops (rrt.py:418-437, 498-548, 690-748) + go2goal (rrt.py:284-332) ---------- */
/*
 * Runs nplans independent plans, one thread block each, tree and bit grid resident on chip.
 *   d_bits     nworlds tiled bit grids (rrtk_pack_grid)
 *   d_plans    nplans descriptors
 *   d_samples  nplans x n x (x, y) int16: sample i of plan p is what sample_all_free returns in
 *              iteration i (rrt.py:421,502,696)
 *   d_balls    informed only: nplans x n x 2 doubles, the unitball() point (rrt.py:579-587) used in
 *              iteration i if that iteration samples the ellipse; may be NULL for other kinds.
 *              Informed with d_balls == NULL is a probe run: each plan stops at its first solution
 *              vertex (RRTK_STAT_FIRST_SOL_ITER tells the caller where the ellipse phase starts)
 *   outputs, (n + 1) rows per plan -- row j is the goal vertex when connected (rrt.py:319-325):
 *   d_pts      int16 (x, y); rows the reference leaves unfilled hold (-32768, -32768)
 *   d_cost     float64 cost-to-come (vcosts); +inf in unfilled rows
 *   d_parent   int32 parent vertex; -1 for the root and unfilled rows
 *   d_stats    RRTK_STAT_COUNT int64 per plan
 *   d_ell_c    informed only (else NULL): d_ell_c[p*(n+1) + j] = cbest of the last ellipse sample
 *              drawn while the tree had j vertices (rrt.py:698-701), NaN where none
 * r_rewire / r_goal as in the constructors (rrt.py:454-464, 563-577).  `threads` = block size
 * (0 = library default).
 */
int rrtk_plan_batch(int kind, const uint32_t *d_bits, int W, int H, const rrtk_plan_desc *d_plans,
                    int nplans, int n, double r_rewire, double r_goal, const int16_t *d_samples,
                    const double *d_balls, int16_t *d_pts, double *d_cost, int32_t *d_parent,
                    int64_t *d_stats, double *d_ell_c, int threads, void *stream);

/* Which plan kernel rrtk_plan_batch runs for this shape on the current device: "grid" (RRTStandard / RRTStar, n >= 256,
 * tree entries fit one word: near / within from spatial buckets of the pre-known samples), "scan" (brute-force packed-key scan)
 * or "wide" (32-bit distances, any grid); "" without a device.  The trees are the same whichever runs. */
const char *rrtk_plan_kernel(int kind, int W, int H, int n, int threads);

/* shared memory one plan block needs and how many blocks fit on one SM (for sizing / reporting) */
int rrtk_plan_footprint(int kind, int W, int H, int n, int threads, int *smem_bytes, int *blocks_per_sm);

/* root -> goal vertex paths (RRT.route2gv, rrt.py:87-107 on a tree = parent walk): d_path gets up
 * to cap vertex ids per plan, root first; d_len the path length (0 if vgoal has no parent chain) */
int rrtk_extract_paths(const int32_t *d_parent, const int64_t *d_stats, int nplans, int n, int cap,
                       int32_t *d_path, int32_t *d_len, void *stream);

/* The same walk, returning what a caller of the reference ends up holding for a plan (rrt.py:87-129): vertex ids
 * root -> goal (route2gv), their points (the sequence vertices_as_ndarray pairs up into segments) and the path cost
 * (vcosts[vgoal]; 0 with a one-vertex path when the goal was not connected).  Rows are padded to cap entries with
 * -1 / (-32768, -32768); d_len may exceed cap, in which case that plan's row is left unwritten.  This fixed-size
 * record is what a multi-GPU run gathers (rrtplanner_b200/multigpu.py). */
int rrtk_extract_paths_xy(const int32_t *d_parent, const int16_t *d_pts, const double *d_cost, const int64_t *d_stats,
                          int nplans, int n, int cap, int32_t *d_path, int16_t *d_xy, int32_t *d_len,
                          double *d_path_cost, void *stream);

/* ---- K8: planners the reference advertises but does not ship ---------------------------------------- */
/*
 * README.md:12,18-19 of the reference lists a "Dubins Primitive Module", a "Dubins Vehicle RRT Planner" and a
 * "Dubins Vehicle RRT(star) Planner"; none of them exists in its tree, and its RRT* rewire block (rrt.py:532-546)
 * can never fire (it compares cost(vn -> xnew) with vcosts[vn]).  These entry points supply them.  There is no
 * reference behaviour to match: the specification is oracle/rewire_oracle.c (parity UNPINNED), except that
 * model EUCLID with rewire = 0 reproduces rrtk_plan_batch / the reference's RRTStandard and RRTStar trees exactly.
 *
 *   vertex       (x, y, h): cell and heading index h in [0, nheadings), angle h * 2 pi / nheadings
 *   edge length  EUCLID: straight line (rrt.py:70-78);  DUBINS: shortest of LSL RSR LSR RSL RLR LRL at turning
 *                radius rho (cells), first word on ties, in IEEE double with the specification's own atan2/sin/cos
 *   edge test    EUCLID: rrt.py:183-229 walked parent -> child;  DUBINS: path points every ds cells, rounded to
 *                the nearest cell, plus the end cell; leaving the grid blocks
 *   loop         rrt.py:498-548 with nearest / within Euclidean on (x, y); rewire != 0 adds, for every member vn
 *                of the radius set in ascending order with  cost[vnew] + len(vnew -> vn) < cost[vn]  and a free
 *                edge: parent[vn] = vnew and the costs of vn's subtree recomputed from the edge lengths
 *   informed     (cfg.informed, RRTStarInformed.plan rrt.py:690-748 with a rewire that fires): once a vertex within
 *                r_goal of the goal exists, the (x, y) of iteration i is the ellipse point (rrt.py:589-625, rotation in
 *                rrtk_plan_desc.rot) for c = cost of the cheapest solution vertex (first one on ties, rrt.py:627-633;
 *                costs as lowered by every rewire so far) + its distance to the goal, and unit-disc draw balls[i]
 */
typedef enum { RRTK_MODEL_EUCLID = 0, RRTK_MODEL_DUBINS = 1 } rrtk_model;

typedef struct {
    int32_t model;           /* rrtk_model */
    int32_t star;            /* 0: parent = nearest vertex (RRT)   1: choose parent within r_rewire (RRT*) */
    int32_t rewire;          /* 0: none (what the reference computes)   1: rewire as specified above (needs star) */
    int32_t nheadings;       /* DUBINS: 1 .. 255 heading values */
    double r_rewire;
    double rho;              /* DUBINS: turning radius in cells, 0 < rho <= 16384 */
    double ds;               /* DUBINS: arc-length step of the collision samples in cells, 0.05 <= ds <= 16384 */
    const void *dubins_table; /* DUBINS, optional (NULL = none): DEVICE memo made by rrtk_dubins_table_build for the same
                                nheadings and rho; edges whose |dx|, |dy| <= table_radius are looked up instead of evaluated */
    int32_t table_radius;
    int32_t informed;        /* 1: the informed sampling rule of rrt.py:690-701,744-745 on top of the loop (below) */
    double r_goal;           /* informed: accepted vertices closer than this to the goal (Euclidean, strict) are solution vertices */
    const double *balls;     /* informed: nplans x n x (x, y) unit-disc draws (rrt.py:579-587), row i used by iteration i; NULL = probe
                                run that stops at the first solution vertex.  DEVICE memory for rrtk_plan2_batch, HOST memory for
                                rrtk_ctx_plan2 / rrtk_ctx_plan2_worlds (the call uploads it) */
    double *ell_c;           /* informed, optional output: nplans x (n + 1), entry j = the budget c of the last ellipse sample drawn
                                while the tree had j vertices (rrt.py:701), NaN elsewhere.  DEVICE / HOST as for balls */
} rrtk_plan2_cfg;

/* statistics slots rrtk_plan2_batch writes (RRTK_STAT_COUNT int64 per plan; J / VGOAL / FOUND / CHECKS as above) */
enum {
    RRTK_STAT2_ACCEPTED = 4,   /* accepted samples */
    RRTK_STAT2_REWIRES,        /* rewire operations applied */
    RRTK_STAT2_PROPAGATED,     /* descendant costs recomputed after rewires */
    RRTK_STAT2_RING_MEMBERS,   /* sum over accepted iterations of |within(r_rewire)| */
    RRTK_STAT2_LEN_EVALS,      /* edge lengths evaluated on the device (parallel form) */
    RRTK_STAT2_OVERFLOW,       /* 1: a radius set exceeded the kernel's 1024-entry list; the plan is INVALID */
    RRTK_STAT2_ELL_ITERS,      /* informed: iterations whose sample came from the ellipse */
    RRTK_STAT2_FIRST_SOL       /* informed: iteration that accepted the first solution vertex, -1 = none */
};

/* bytes of device scratch rrtk_plan2_batch needs for nplans plans of n iterations */
size_t rrtk_plan2_scratch_bytes(int nplans, int n);

/*
 * nplans independent plans, one thread block each.  Plan p starts at (start_x, start_y, heading reserved[0]) and
 * ends at (goal_x, goal_y, heading reserved[1]) of its descriptor (headings ignored by EUCLID).
 *   d_samples  nplans x n x (x, y) int16 as for rrtk_plan_batch;  d_heads  nplans x n uint8 heading of sample i
 *              (DUBINS; may be NULL = heading 0)
 *   outputs, (n + 1) rows per plan, row j = goal vertex when connected:
 *   d_pts int16 (x, y) (-32768 unfilled), d_head uint8 (255 unfilled), d_cost / d_elen float64 cost-to-come and
 *   length of the edge from the parent (+inf unfilled), d_parent int32 (-1 root / unfilled), d_stats int64.
 * threads: 0 (default 256), 128 or 256.  n <= 65534.
 */
int rrtk_plan2_batch(const rrtk_plan2_cfg *cfg, const uint32_t *d_bits, int W, int H, const rrtk_plan_desc *d_plans,
                     int nplans, int n, const int16_t *d_samples, const uint8_t *d_heads, int16_t *d_pts, uint8_t *d_head,
                     double *d_cost, double *d_elen, int32_t *d_parent, int64_t *d_stats, void *d_scratch, int threads,
                     void *stream);
int rrtk_plan2_footprint(int n, int threads, int *smem_bytes, int *blocks_per_sm);

/* Memo of the Dubins primitive: with integer cells and indexed headings the shortest path depends only on
 * (dx, dy, h0, h1), so all of them with |dx|, |dy| <= radius fit a table (radius 50, 16 headings: 2.6 M entries, 86 MB,
 * the 21 MB of lengths stay L2-resident) that every plan of a batch shares; the entries are what rrtk_dubins_paths
 * returns, bit for bit.  rrtk_ctx_plan2 builds and caches one on its own. */
size_t rrtk_dubins_table_bytes(int radius, int nheadings);
int rrtk_dubins_table_build(int radius, int nheadings, double rho, void *d_table, void *stream);

/* Dubins primitive, batched.  d_q: nq x (x0, y0, h0, x1, y1, h1) int32.  Outputs (each optional): d_word 0..5 =
 * LSL RSR LSR RSL RLR LRL, d_tpq nq x 3 segment lengths in units of rho, d_len path length in cells. */
int rrtk_dubins_paths(const int32_t *d_q, int64_t nq, int nheadings, double rho, int32_t *d_word, double *d_tpq,
                      double *d_len, void *stream);
/* sampled collision test of the shortest path of each query (the edge test above); d_world optional per query */
int rrtk_dubins_collision(const uint32_t *d_bits, int W, int H, const int32_t *d_q, const int32_t *d_world, int64_t nq,
                          int nheadings, double rho, double ds, uint8_t *d_free, void *stream);
/* poses (x, y, theta) of each query's shortest path every ds cells: d_xyth nq x cap x 3, d_count[q] = number of
 * poses the path has (floor(len / ds) + 1; only the first cap are stored) */
int rrtk_dubins_sample(const int32_t *d_q, int64_t nq, int nheadings, double rho, double ds, int cap, double *d_xyth,
                       int32_t *d_count, void *stream);

/* ---- host-buffer entry points (the call a Python planner object makes; copies inside) ------------ */
typedef struct rrtk_ctx rrtk_ctx;    /* owns device scratch; one per planner object / thread */
int rrtk_create(rrtk_ctx **out);
int rrtk_destroy(rrtk_ctx *ctx);

/* upload nworlds (W,H) uint8 grids, pack them (K0) and build the free-space index; replaces the
 * state RRT.__init__ / RRT.set_og keep (rrt.py:64-65, 261-272).  h_nfree (optional) receives the
 * number of free cells per world. */
int rrtk_ctx_set_grids(rrtk_ctx *ctx, const uint8_t *h_og, int nworlds, int W, int H, int32_t *h_nfree);

/* host-buffer form of rrtk_inflate_grid for ONE (W,H) uint8 source grid: h_out receives nout inflated uint8
 * grids (one per hole triple in h_holes, or a single one without holes when h_holes is NULL and nout = 1) */
int rrtk_ctx_inflate(rrtk_ctx *ctx, const uint8_t *h_og, int W, int H, int iterations, const int32_t *h_holes, int nout,
                     uint8_t *h_out);

/* full plan() from host memory: H2D of descriptors (+ samples / balls / PCG64 states), K7, D2H of
 * the trees.  Exactly one of h_samples / h_state must be non-NULL (explicit stream vs. seed mode).
 * Output arrays as in rrtk_plan_batch but in host memory. */
int rrtk_ctx_plan(rrtk_ctx *ctx, int kind, const rrtk_plan_desc *h_plans, int nplans, int n,
                  double r_rewire, double r_goal, const int16_t *h_samples, const uint64_t *h_state,
                  const double *h_balls, int16_t *h_pts, double *h_cost, int32_t *h_parent,
                  int64_t *h_stats, double *h_ell_c);

/* rrtk_ctx_set_grids + rrtk_ctx_plan in one call, pipelined: plans (ordered by world index) are
 * processed in chunks of chunk_plans (0 = two plan blocks per SM, the first chunk one per SM) on rotating plan streams
 * between one preparation and one output stream, so the upload of one chunk's grids and the download of another's trees
 * overlap the kernels; give pinned host buffers for the copies to be asynchronous.  The worlds are not kept in the
 * context afterwards.  Seed mode (h_state) on a world without a free cell is an error as in rrtk_ctx_plan
 * (RRTK_ERR_INVALID; found on the device, so reported when the call returns: the outputs then mean nothing). */
int rrtk_ctx_plan_worlds(rrtk_ctx *ctx, int kind, const uint8_t *h_og, int nworlds, int W, int H,
                         const rrtk_plan_desc *h_plans, int nplans, int n, double r_rewire, double r_goal,
                         const int16_t *h_samples, const uint64_t *h_state, const double *h_balls,
                         int16_t *h_pts, double *h_cost, int32_t *h_parent, int64_t *h_stats, double *h_ell_c,
                         int chunk_plans);

/* The same pipeline with the two ends a batch caller can choose (what `set_og` + `plan` + `route2gv` /
 * `vertices_as_ndarray` amount to for many plans, rrt.py:261-272, 87-129):
 *   RRTK_IN_BITS    h_grids holds tiled bit grids (rrtk_grid_words(W,H) uint32 per world, the layout at the top of
 *                   this file; rrtk_pack_grid_host makes them) instead of uint8 cells: 1/8 of the upload
 *   RRTK_OUT_TREES  download every tree (h_pts, h_cost, h_parent, and h_ell_c for informed plans)
 *   RRTK_OUT_PATHS  download the path record of every plan as rrtk_extract_paths_xy writes it (path_cap entries per
 *                   plan in h_path / h_xy, h_len, h_path_cost): ~2 KB per plan instead of 16 B per tree row
 * h_stats always comes back.  Output pointers of a mode that is not requested may be NULL.  On an error after the first
 * copy was enqueued the call drains every stream before it returns, so no transfer is still writing into the caller's
 * buffers.  RRTK_PIPE_TRACE=1 in the environment prints the device time stamps of every chunk's stages to stderr.
 *   RRTK_SEED_BALLS informed plans in seed mode draw their ellipse phase from the plan's own generator, as a seeded
 *                   RRTStarInformed object does (rrt.py:85, 240, 579-587): per chunk, sample streams -> probe launch ->
 *                   rrtk_ball_streams on the probe's statistics -> full launch.  Needs h_state, kind RRTK_INFORMED and
 *                   h_balls == NULL (RRTK_ERR_INVALID otherwise, before any device work); nothing per iteration is uploaded.
 *                   The descriptors carry the rotation as before; a plan whose rotation is not finite (start == goal)
 *                   and that reaches the ellipse phase makes the call fail with RRTK_ERR_INVALID naming it (found on the
 *                   device, so reported when the call returns).  rrtk_ctx_plan2_worlds takes the flag with cfg->informed
 *                   and cfg->balls == NULL. */
#define RRTK_IN_BITS 1
#define RRTK_OUT_TREES 2
#define RRTK_OUT_PATHS 4
#define RRTK_SEED_BALLS 8
int rrtk_ctx_plan_worlds2(rrtk_ctx *ctx, int kind, const void *h_grids, int nworlds, int W, int H,
                          const rrtk_plan_desc *h_plans, int nplans, int n, double r_rewire, double r_goal,
                          const int16_t *h_samples, const uint64_t *h_state, const double *h_balls, int flags,
                          int path_cap, int16_t *h_pts, double *h_cost, int32_t *h_parent, int64_t *h_stats,
                          double *h_ell_c, int32_t *h_path, int16_t *h_xy, int32_t *h_len, double *h_path_cost,
                          int chunk_plans);

/* `np.random.default_rng(seed)` (rrt.py:85) -> the PCG64 start state the seed modes take: {state_hi, state_lo, inc_hi,
 * inc_lo} per seed, by numpy's published SeedSequence + pcg_setseq_128_srandom_r path.  Plain CPU code, no device needed. */
int rrtk_seed_states(const uint64_t *h_seeds, int nseeds, uint64_t *h_state);

/* K0 on the host, for callers that keep their worlds packed (`og[x, y] != 0`, rrt.py:218, one bit per cell in the
 * tiled layout; cells outside the grid are set).  Plain CPU loop, no device needed. */
int rrtk_pack_grid_host(const uint8_t *h_og, int nworlds, int W, int H, uint32_t *h_bits);

/* the sample stream a planner seeded with h_state would draw (seed mode of rrtk_ctx_plan, exposed
 * so RRT.sample_all_free can be served from the same generator) */
int rrtk_ctx_samples(rrtk_ctx *ctx, const rrtk_plan_desc *h_plans, int nplans, int n, const uint64_t *h_state,
                     int16_t *h_samples);

/* host-buffer forms of K1-K3 on the context's world `world` */
int rrtk_ctx_collision(rrtk_ctx *ctx, int world, const int32_t *h_segs, int64_t nseg, uint8_t *h_free,
                       int32_t *h_cells);
int rrtk_ctx_nearest(rrtk_ctx *ctx, const int32_t *h_pts, int npts, const int32_t *h_queries, int nq,
                     int32_t *h_idx, int64_t *h_d2);
int rrtk_ctx_within(rrtk_ctx *ctx, const int32_t *h_pts, int npts, const int32_t *h_queries, int nq,
                    double r, int cap, int32_t *h_out, int32_t *h_len);
int rrtk_ctx_near_order(rrtk_ctx *ctx, const int32_t *h_pts, int npts, int qx, int qy, int32_t *h_perm);
int rrtk_ctx_nearest_f64(rrtk_ctx *ctx, const double *h_pts, int npts, const double *h_queries, int nq,
                         int32_t *h_idx, double *h_dist);
int rrtk_ctx_within_f64(rrtk_ctx *ctx, const double *h_pts, int npts, const double *h_queries, int nq,
                        double r, int cap, int32_t *h_out, int32_t *h_len);
int rrtk_ctx_near_order_f64(rrtk_ctx *ctx, const double *h_pts, int npts, double qx, double qy, int32_t *h_perm);

/* host-buffer forms of K8 (rrtk_plan2_batch on the context's worlds; exactly one of h_samples / h_state as for
 * rrtk_ctx_plan) and of the Dubins primitive */
int rrtk_ctx_plan2(rrtk_ctx *ctx, const rrtk_plan2_cfg *cfg, const rrtk_plan_desc *h_plans, int nplans, int n,
                   const int16_t *h_samples, const uint64_t *h_state, const uint8_t *h_heads, int16_t *h_pts,
                   uint8_t *h_head, double *h_cost, double *h_elen, int32_t *h_parent, int64_t *h_stats);
/* rrtk_ctx_plan2 with the worlds in the same call, chunked and pipelined like rrtk_ctx_plan_worlds2 (same flags, same
 * ordering rule for plans, same meaning of h_grids / h_path / h_xy / h_len / h_path_cost; set_og + plan of
 * rrt.py:261-272,498-548 for a batch of K8 plans).  RRTK_OUT_TREES additionally fills h_head and h_elen; h_path_head
 * (optional, RRTK_OUT_PATHS) receives nplans x path_cap uint8 headings of the path vertices (255 past the end), which a
 * Dubins path needs beside its points.  chunk_plans <= 0: one plan per SM and chunk. */
int rrtk_ctx_plan2_worlds(rrtk_ctx *ctx, const rrtk_plan2_cfg *cfg, const void *h_grids, int nworlds, int W, int H,
                          const rrtk_plan_desc *h_plans, int nplans, int n, const int16_t *h_samples,
                          const uint64_t *h_state, const uint8_t *h_heads, int flags, int path_cap, int16_t *h_pts,
                          uint8_t *h_head, double *h_cost, double *h_elen, int32_t *h_parent, int64_t *h_stats,
                          int32_t *h_path, int16_t *h_xy, uint8_t *h_path_head, int32_t *h_len, double *h_path_cost,
                          int chunk_plans);
int rrtk_ctx_dubins_paths(rrtk_ctx *ctx, const int32_t *h_q, int64_t nq, int nheadings, double rho, int32_t *h_word,
                          double *h_tpq, double *h_len);
int rrtk_ctx_dubins_collision(rrtk_ctx *ctx, int world, const int32_t *h_q, int64_t nq, int nheadings, double rho,
                              double ds, uint8_t *h_free);
int rrtk_ctx_dubins_sample(rrtk_ctx *ctx, const int32_t *h_q, int64_t nq, int nheadings, double rho, double ds, int cap,
                           double *h_xyth, int32_t *h_count);

#ifdef __cplusplus
}
#endif
#endif /* RRTK_H */
