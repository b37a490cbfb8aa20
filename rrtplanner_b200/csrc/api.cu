// extern "C" surface of librrtk.so (declared in include/rrtk.h): argument checks, device info,
// the host-buffer context, and thin forwards to the kernel launchers.
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <chrono>
#include <vector>

#include "common.cuh"

namespace rrtk {

static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
int cuda_fail(cudaError_t e, const char *what)
{
    set_error("CUDA error %d (%s) in %s", (int)e, cudaGetErrorString(e), what);
    return e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver ? RRTK_ERR_NODEVICE : RRTK_ERR_CUDA;
}

// launchers implemented in the other translation units
int pack_launch(const uint8_t *, int, int, int, uint32_t *, cudaStream_t);
int free_rows_launch(const uint32_t *, int, int, int, int32_t *, cudaStream_t);
int worlds_launch(const int32_t *, int, int, int, int, int32_t *, uint8_t *, cudaStream_t);
int collision_launch(const uint32_t *, int, int, const int32_t *, const int32_t *, int64_t, uint8_t *, int32_t *, int, int,
                     cudaStream_t);
int clearance_launch(const uint32_t *, int, int, int, int, uint8_t *, uint32_t *, cudaStream_t);
int clearance_dir_launch(const uint32_t *, int, int, int, int, uint8_t *, cudaStream_t);
int clearance_dir16_launch(const uint32_t *, int, int, int, int, uint8_t *, cudaStream_t);
int collision_cf_launch(const uint8_t *, int, int, const int32_t *, const int32_t *, int, int64_t, uint8_t *, int32_t *, int, cudaStream_t);
int unpack_launch(const uint32_t *, int, int, int, uint8_t *, cudaStream_t);
int inflate_launch(const uint32_t *, int, int, int, int, const int32_t *, int, uint32_t *, uint32_t *, cudaStream_t);
int nearest_launch(const int32_t *, int, const int32_t *, const int32_t *, int, int32_t *, int64_t *, cudaStream_t);
int nearest_launch_f64(const double *, int, const double *, const int32_t *, int, int32_t *, double *, cudaStream_t);
int within_launch(const int32_t *, int, const int32_t *, const int32_t *, int, double, int, int32_t *, int32_t *, cudaStream_t);
int within_launch_f64(const double *, int, const double *, const int32_t *, int, double, int, int32_t *, int32_t *, cudaStream_t);
int dist2_launch(const int32_t *, int, int, int, int64_t *, cudaStream_t);
int dist_launch_f64(const double *, int, double, double, double *, cudaStream_t);
int argsort_launch(const int64_t *, int, int32_t *, void *, size_t, cudaStream_t);
size_t argsort_scratch(int);
int sample_streams_launch(const uint32_t *, const int32_t *, int, int, const rrtk_plan_desc *, int, const uint64_t *, int,
                          int16_t *, int, cudaStream_t, uint64_t * = nullptr, uint32_t * = nullptr);
int ball_streams_launch(const int32_t *, int, const rrtk_plan_desc *, int, int, const uint64_t *, const uint32_t *, const int64_t *, int,
                        double *, uint64_t *, uint32_t *, cudaStream_t);
int plan_launch(int, const uint32_t *, int, int, const rrtk_plan_desc *, int, int, double, double, const int16_t *,
                const double *, int16_t *, double *, int32_t *, int64_t *, double *, int, int, int, cudaStream_t);
int plan_footprint(int, int, int, int, int, int, int, int *, int *);
const char *plan_kernel_name(int, int, int, int, int, int, int);
int paths_launch(const int32_t *, const int64_t *, int, int, int, int32_t *, int32_t *, cudaStream_t);
int path_heads_launch(const int32_t *, const uint8_t *, int, int, int, uint8_t *, cudaStream_t);
int paths_xy_launch(const int32_t *, const int16_t *, const double *, const int64_t *, int, int, int, int32_t *, int16_t *, int32_t *,
                    double *, cudaStream_t);
int plan2_launch(const rrtk_plan2_cfg &, const uint32_t *, int, int, const rrtk_plan_desc *, int, int, const int16_t *, const uint8_t *,
                 int16_t *, uint8_t *, double *, double *, int32_t *, int64_t *, void *, int, int, cudaStream_t);
size_t plan2_scratch_bytes(int, int);
int plan2_footprint(int, int, int, int, int *, int *);
int dubins_paths_launch(const int32_t *, int64_t, int, double, int32_t *, double *, double *, cudaStream_t);
size_t dubins_table_bytes(int, int);
int dubins_table_launch(int, int, double, void *, int, cudaStream_t);
int l2_read_launch(const void *, size_t, int, int, uint32_t *, cudaStream_t);
int smem_read_launch(int, int, int, uint32_t *, cudaStream_t);
int dubins_walk_launch(const uint32_t *, int, int, const int32_t *, const int32_t *, int64_t, int, double, double, uint8_t *, int,
                       double *, int32_t *, cudaStream_t);

struct DevInfo { int dev = -1, sms = 0, optin = 0, sm_smem = 0; };
static thread_local DevInfo g_dev;

static int dev_info(DevInfo **out)
{
    int dev = 0;
    RRTK_CUDA(cudaGetDevice(&dev));
    if (g_dev.dev != dev) {
        RRTK_CUDA(cudaDeviceGetAttribute(&g_dev.sms, cudaDevAttrMultiProcessorCount, dev));
        RRTK_CUDA(cudaDeviceGetAttribute(&g_dev.optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
        RRTK_CUDA(cudaDeviceGetAttribute(&g_dev.sm_smem, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev));
        g_dev.dev = dev;
    }
    *out = &g_dev;
    return RRTK_OK;
}

static int check_grid_dims(int W, int H, int limit)
{
    if (W < 1 || H < 1 || W > limit || H > limit) {
        set_error("grid size (%d, %d) out of range [1, %d]", W, H, limit);
        return RRTK_ERR_INVALID;
    }
    return RRTK_OK;
}
#define RRTK_REQUIRE(cond, msg)                 \
    do {                                        \
        if (!(cond)) {                          \
            rrtk::set_error("%s", msg);         \
            return RRTK_ERR_INVALID;            \
        }                                       \
    } while (0)
#define RRTK_TRY(call)                  \
    do {                                \
        int rc_ = (call);               \
        if (rc_ != RRTK_OK) return rc_; \
    } while (0)

}  // namespace rrtk

using namespace rrtk;

// ---- device-side growable buffer used by the host-buffer context ---------------------------------
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes)
    {
        if (bytes <= cap) return RRTK_OK;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        RRTK_CUDA(cudaMalloc(&p, bytes));
        cap = bytes;
        return RRTK_OK;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T *as() { return reinterpret_cast<T *>(p); }
};

// One stage of the chunked upload / plan / download pipeline of rrtk_ctx_plan_worlds2 / rrtk_ctx_plan2_worlds.
// Streams: ONE preparation stream for all chunks (uploads, packing, free-space index, sampler) and ONE output stream
// (path extraction, downloads), both of the highest priority so that their short kernels get SM resources ahead of the
// pending plan blocks (a plan kernel leaves no free registers on an SM it fills), plus one plan stream per slot.  That is
// 2 + kPipeSlots streams: with the context's own stream they fit the 8 hardware queues of a default CUDA context
// (CUDA_DEVICE_MAX_CONNECTIONS), where streams that share a queue serialise behind each other -- with 16 streams a chunk's
// plan kernel waited for the chunk four before it to finish entirely (RRTK_PIPE_TRACE=1 prints the time stamps).
struct PipeSlot {
    cudaStream_t stream = nullptr;              // the chunk's plan kernel
    cudaEvent_t ready = nullptr, planned = nullptr, done = nullptr;   // inputs on the device / plan kernel finished / outputs on the host
    DevBuf og, bits, rowcum, plans, samples, state, balls, pts, cost, parent, stats, ell;
    DevBuf path, xy, len, pcost;                // path records (RRTK_OUT_PATHS)
    DevBuf heads, head_out, elen, scratch2, phead;   // K8 chunks (rrtk_ctx_plan2_worlds)
    std::vector<rrtk_plan_desc> desc;
};
constexpr int kPipeSlots = 5;

struct rrtk_ctx {
    cudaStream_t stream = nullptr;
    int W = 0, H = 0, nworlds = 0;
    std::vector<int32_t> nfree;                 // free cells per world (a world without any cannot be sampled: rrt.py:240)
    DevBuf og, bits, rowcum;                    // worlds
    DevBuf plans, samples, state, balls;        // plan inputs
    DevBuf pts, cost, parent, stats, ell;       // plan outputs
    DevBuf a, b, c, d, e;                       // query scratch
    DevBuf heads, head_out, elen, scratch2;     // K8 (rrtk_ctx_plan2)
    DevBuf dtable;                              // memo of the Dubins primitive, valid for (dt_R, dt_NH, dt_rho)
    int dt_R = 0, dt_NH = 0;
    double dt_rho = 0.0;
    PipeSlot pipe[kPipeSlots];
    cudaStream_t pipe_prep = nullptr, pipe_post = nullptr;
    int32_t *pin_nfree = nullptr;               // pinned: free cells per world of a pipelined call (seed mode checks them)
    size_t pin_nfree_cap = 0;
};

extern "C" {

int rrtk_version(void) { return RRTK_VERSION; }
const char *rrtk_last_error(void) { return g_err; }

int rrtk_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}
int rrtk_set_device(int device)
{
    RRTK_CUDA(cudaSetDevice(device));
    return RRTK_OK;
}
int rrtk_device_info(int *sm_count, int *smem_optin_bytes)
{
    DevInfo *d;
    RRTK_TRY(dev_info(&d));
    if (sm_count) *sm_count = d->sms;
    if (smem_optin_bytes) *smem_optin_bytes = d->optin;
    return RRTK_OK;
}

size_t rrtk_grid_words(int W, int H) { return (W < 1 || H < 1) ? 0 : grid_words(W, H); }

int rrtk_pack_grid(const uint8_t *d_og, int nworlds, int W, int H, uint32_t *d_bits, void *stream)
{
    RRTK_REQUIRE(d_og && d_bits && nworlds >= 0, "rrtk_pack_grid: null pointer or negative count");
    RRTK_TRY(check_grid_dims(W, H, 32768));
    if (nworlds == 0) return RRTK_OK;
    return pack_launch(d_og, nworlds, W, H, d_bits, (cudaStream_t)stream);
}

int rrtk_unpack_grid(const uint32_t *d_bits, int nworlds, int W, int H, uint8_t *d_og, void *stream)
{
    RRTK_REQUIRE(d_og && d_bits && nworlds >= 0, "rrtk_unpack_grid: null pointer or negative count");
    RRTK_TRY(check_grid_dims(W, H, 32768));
    return unpack_launch(d_bits, nworlds, W, H, d_og, (cudaStream_t)stream);
}

int rrtk_inflate_grid(const uint32_t *d_bits, int nworlds, int W, int H, int iterations, const int32_t *d_holes,
                      int nout, uint32_t *d_out, uint32_t *d_scratch, void *stream)
{
    RRTK_REQUIRE(d_bits && d_out && d_scratch && nworlds >= 0 && iterations >= 0, "rrtk_inflate_grid: null pointer or negative count");
    RRTK_REQUIRE(nout >= nworlds, "rrtk_inflate_grid: nout must be at least nworlds");
    RRTK_REQUIRE(d_out != d_bits && d_scratch != d_bits && d_out != d_scratch, "rrtk_inflate_grid: buffers must not alias");
    RRTK_TRY(check_grid_dims(W, H, 32768));
    if (nworlds == 0) return RRTK_OK;
    return inflate_launch(d_bits, nworlds, W, H, iterations, d_holes, nout, d_out, d_scratch, (cudaStream_t)stream);
}

int rrtk_free_rows(const uint32_t *d_bits, int nworlds, int W, int H, int32_t *d_rowcum, void *stream)
{
    RRTK_REQUIRE(d_bits && d_rowcum && nworlds >= 0, "rrtk_free_rows: null pointer or negative count");
    RRTK_TRY(check_grid_dims(W, H, 32768));
    if (nworlds == 0) return RRTK_OK;
    return free_rows_launch(d_bits, nworlds, W, H, d_rowcum, (cudaStream_t)stream);
}

int rrtk_gen_worlds(const int32_t *d_seeds, int nworlds, int W, int H, int thresh_permille, int32_t *d_scratch,
                    uint8_t *d_og, void *stream)
{
    RRTK_REQUIRE(d_seeds && d_scratch && d_og, "rrtk_gen_worlds: null pointer");
    RRTK_REQUIRE(nworlds >= 0 && nworlds <= 65535, "rrtk_gen_worlds: nworlds must be in [0, 65535] per call");
    RRTK_TRY(check_grid_dims(W, H, 16384));
    if (nworlds == 0) return RRTK_OK;
    return worlds_launch(d_seeds, nworlds, W, H, thresh_permille, d_scratch, d_og, (cudaStream_t)stream);
}

int rrtk_collision_segments(const uint32_t *d_bits, int W, int H, const int32_t *d_segs, const int32_t *d_world,
                            int64_t nseg, uint8_t *d_free, int32_t *d_cells, void *stream)
{
    RRTK_REQUIRE(d_bits && (nseg == 0 || (d_segs && d_free)) && nseg >= 0, "rrtk_collision_segments: null pointer");
    RRTK_TRY(check_grid_dims(W, H, 32768));
    DevInfo *d;
    RRTK_TRY(dev_info(&d));
    return collision_launch(d_bits, W, H, d_segs, d_world, nseg, d_free, d_cells, d->sms, d->optin, (cudaStream_t)stream);
}

int rrtk_clearance_field(const uint32_t *d_bits, int nworlds, int W, int H, int cap, uint8_t *d_clear, uint32_t *d_scratch, void *stream)
{
    RRTK_REQUIRE(d_bits && d_clear && d_scratch && nworlds >= 0, "rrtk_clearance_field: null pointer or negative count");
    RRTK_REQUIRE(cap >= 2 && cap <= 255, "rrtk_clearance_field: cap must be in [2, 255]");
    RRTK_TRY(check_grid_dims(W, H, 32768));
    if (nworlds == 0) return RRTK_OK;
    return clearance_launch(d_bits, nworlds, W, H, cap, d_clear, d_scratch, (cudaStream_t)stream);
}

int rrtk_collision_segments_cf(const uint8_t *d_clear, int W, int H, const int32_t *d_segs, const int32_t *d_world, int64_t nseg,
                               uint8_t *d_free, int32_t *d_cells, void *stream)
{
    RRTK_REQUIRE(nseg >= 0 && (nseg == 0 || (d_clear && d_segs && d_free)), "rrtk_collision_segments_cf: bad argument");
    RRTK_TRY(check_grid_dims(W, H, 32768));
    DevInfo *d;
    RRTK_TRY(dev_info(&d));
    return collision_cf_launch(d_clear, W, H, d_segs, d_world, 1, nseg, d_free, d_cells, d->sms, (cudaStream_t)stream);
}

int rrtk_clearance_field_dir(const uint32_t *d_bits, int nworlds, int W, int H, int cap, uint8_t *d_clear8, void *stream)
{
    RRTK_REQUIRE(d_bits && d_clear8 && nworlds >= 0, "rrtk_clearance_field_dir: null pointer or negative count");
    RRTK_REQUIRE(cap >= 2 && cap <= 255, "rrtk_clearance_field_dir: cap must be in [2, 255]");
    RRTK_TRY(check_grid_dims(W, H, 32768));
    if (nworlds == 0) return RRTK_OK;
    return clearance_dir_launch(d_bits, nworlds, W, H, cap, d_clear8, (cudaStream_t)stream);
}

int rrtk_collision_segments_cfd(const uint8_t *d_clear8, int W, int H, const int32_t *d_segs, const int32_t *d_world, int64_t nseg,
                                uint8_t *d_free, int32_t *d_cells, void *stream)
{
    RRTK_REQUIRE(nseg >= 0 && (nseg == 0 || (d_clear8 && d_segs && d_free)), "rrtk_collision_segments_cfd: bad argument");
    RRTK_TRY(check_grid_dims(W, H, 32768));
    DevInfo *d;
    RRTK_TRY(dev_info(&d));
    return collision_cf_launch(d_clear8, W, H, d_segs, d_world, 8, nseg, d_free, d_cells, d->sms, (cudaStream_t)stream);
}

int rrtk_clearance_field_dir16(const uint32_t *d_bits, int nworlds, int W, int H, int cap, uint8_t *d_clear16, void *stream)
{
    RRTK_REQUIRE(d_bits && d_clear16 && nworlds >= 0, "rrtk_clearance_field_dir16: null pointer or negative count");
    RRTK_REQUIRE(cap >= 2 && cap <= 255, "rrtk_clearance_field_dir16: cap must be in [2, 255]");
    RRTK_TRY(check_grid_dims(W, H, 32768));
    if (nworlds == 0) return RRTK_OK;
    return clearance_dir16_launch(d_bits, nworlds, W, H, cap, d_clear16, (cudaStream_t)stream);
}

int rrtk_collision_segments_cfd16(const uint8_t *d_clear16, int W, int H, const int32_t *d_segs, const int32_t *d_world, int64_t nseg,
                                  uint8_t *d_free, int32_t *d_cells, void *stream)
{
    RRTK_REQUIRE(nseg >= 0 && (nseg == 0 || (d_clear16 && d_segs && d_free)), "rrtk_collision_segments_cfd16: bad argument");
    RRTK_TRY(check_grid_dims(W, H, 32768));
    DevInfo *d;
    RRTK_TRY(dev_info(&d));
    return collision_cf_launch(d_clear16, W, H, d_segs, d_world, 16, nseg, d_free, d_cells, d->sms, (cudaStream_t)stream);
}

int rrtk_nearest_batch(const int32_t *d_pts, int npts, const int32_t *d_queries, const int32_t *d_count, int nq,
                       int32_t *d_idx, int64_t *d_d2, void *stream)
{
    RRTK_REQUIRE(npts >= 0 && nq >= 0 && (nq == 0 || (d_queries && d_idx)) && (npts == 0 || d_pts), "rrtk_nearest_batch: bad argument");
    return nearest_launch(d_pts, npts, d_queries, d_count, nq, d_idx, d_d2, (cudaStream_t)stream);
}
int rrtk_nearest_batch_f64(const double *d_pts, int npts, const double *d_queries, const int32_t *d_count, int nq,
                           int32_t *d_idx, double *d_dist, void *stream)
{
    RRTK_REQUIRE(npts >= 0 && nq >= 0 && (nq == 0 || (d_queries && d_idx)) && (npts == 0 || d_pts), "rrtk_nearest_batch_f64: bad argument");
    return nearest_launch_f64(d_pts, npts, d_queries, d_count, nq, d_idx, d_dist, (cudaStream_t)stream);
}

int rrtk_within_batch(const int32_t *d_pts, int npts, const int32_t *d_queries, const int32_t *d_count, int nq, double r,
                      int cap, int32_t *d_out, int32_t *d_len, void *stream)
{
    RRTK_REQUIRE(npts >= 0 && nq >= 0 && cap >= 0 && (nq == 0 || (d_queries && d_len && (cap == 0 || d_out))) && (npts == 0 || d_pts),
                 "rrtk_within_batch: bad argument");
    return within_launch(d_pts, npts, d_queries, d_count, nq, r, cap, d_out, d_len, (cudaStream_t)stream);
}
int rrtk_within_batch_f64(const double *d_pts, int npts, const double *d_queries, const int32_t *d_count, int nq, double r,
                          int cap, int32_t *d_out, int32_t *d_len, void *stream)
{
    RRTK_REQUIRE(npts >= 0 && nq >= 0 && cap >= 0 && (nq == 0 || (d_queries && d_len && (cap == 0 || d_out))) && (npts == 0 || d_pts),
                 "rrtk_within_batch_f64: bad argument");
    return within_launch_f64(d_pts, npts, d_queries, d_count, nq, r, cap, d_out, d_len, (cudaStream_t)stream);
}

int rrtk_dist2(const int32_t *d_pts, int npts, int qx, int qy, int64_t *d_d2, void *stream)
{
    RRTK_REQUIRE(npts >= 0 && (npts == 0 || (d_pts && d_d2)), "rrtk_dist2: bad argument");
    return dist2_launch(d_pts, npts, qx, qy, d_d2, (cudaStream_t)stream);
}
int rrtk_dist_f64(const double *d_pts, int npts, double qx, double qy, double *d_dist, void *stream)
{
    RRTK_REQUIRE(npts >= 0 && (npts == 0 || (d_pts && d_dist)), "rrtk_dist_f64: bad argument");
    return dist_launch_f64(d_pts, npts, qx, qy, d_dist, (cudaStream_t)stream);
}
size_t rrtk_argsort_scratch_bytes(int n) { return argsort_scratch(n); }
int rrtk_argsort_i64(const int64_t *d_keys, int n, int32_t *d_perm, void *d_scratch, size_t scratch_bytes, void *stream)
{
    RRTK_REQUIRE(n >= 0 && (n == 0 || (d_keys && d_perm && d_scratch)), "rrtk_argsort_i64: bad argument");
    return argsort_launch(d_keys, n, d_perm, d_scratch, scratch_bytes, (cudaStream_t)stream);
}

int rrtk_sample_streams(const uint32_t *d_bits, const int32_t *d_rowcum, int W, int H, const rrtk_plan_desc *d_plans,
                        int nplans, const uint64_t *d_state, int n, int16_t *d_samples, void *stream)
{
    RRTK_REQUIRE(d_bits && d_rowcum && d_plans && d_state && d_samples && nplans >= 0 && n >= 0, "rrtk_sample_streams: bad argument");
    RRTK_TRY(check_grid_dims(W, H, 16384));
    DevInfo *d;
    RRTK_TRY(dev_info(&d));
    return sample_streams_launch(d_bits, d_rowcum, W, H, d_plans, nplans, d_state, n, d_samples, d->optin, (cudaStream_t)stream);
}

int rrtk_sample_streams_carry(const uint32_t *d_bits, const int32_t *d_rowcum, int W, int H, const rrtk_plan_desc *d_plans,
                              int nplans, uint64_t *d_state, uint32_t *d_carry, int n, int16_t *d_samples, void *stream)
{
    RRTK_REQUIRE(d_bits && d_rowcum && d_plans && d_state && d_carry && d_samples && nplans >= 0 && n >= 0,
                 "rrtk_sample_streams_carry: bad argument");
    RRTK_TRY(check_grid_dims(W, H, 16384));
    DevInfo *d;
    RRTK_TRY(dev_info(&d));
    return sample_streams_launch(d_bits, d_rowcum, W, H, d_plans, nplans, d_state, n, d_samples, d->optin, (cudaStream_t)stream,
                                 d_state, d_carry);
}

int rrtk_ball_streams(const int32_t *d_rowcum, int W, const rrtk_plan_desc *d_plans, int nplans, int n, const uint64_t *d_state,
                      const uint32_t *d_carry, const int64_t *d_first, int first_stride, double *d_balls, uint64_t *d_state_out,
                      uint32_t *d_carry_out, void *stream)
{
    RRTK_REQUIRE(d_rowcum && d_plans && d_state && d_first && d_balls && nplans >= 0 && n >= 1 && first_stride >= 1,
                 "rrtk_ball_streams: bad argument (null pointer, nplans < 0, n < 1 or first_stride < 1)");
    RRTK_TRY(check_grid_dims(W, 1, 16384));
    return ball_streams_launch(d_rowcum, W, d_plans, nplans, n, d_state, d_carry, d_first, first_stride, d_balls, d_state_out, d_carry_out,
                               (cudaStream_t)stream);
}

int rrtk_plan_batch(int kind, const uint32_t *d_bits, int W, int H, const rrtk_plan_desc *d_plans, int nplans, int n,
                    double r_rewire, double r_goal, const int16_t *d_samples, const double *d_balls, int16_t *d_pts,
                    double *d_cost, int32_t *d_parent, int64_t *d_stats, double *d_ell_c, int threads, void *stream)
{
    RRTK_REQUIRE(d_bits && d_plans && d_samples && d_pts && d_cost && d_parent && d_stats, "rrtk_plan_batch: null pointer");
    RRTK_REQUIRE(kind != RRTK_INFORMED || d_ell_c, "rrtk_plan_batch: informed plans need d_ell_c");
    RRTK_REQUIRE(nplans >= 0 && n >= 1 && n <= 65534, "rrtk_plan_batch: need nplans >= 0 and 1 <= n <= 65534");
    RRTK_REQUIRE(r_rewire == r_rewire && r_goal == r_goal, "rrtk_plan_batch: NaN radius");
    RRTK_TRY(check_grid_dims(W, H, 16384));
    if (nplans == 0) return RRTK_OK;
    DevInfo *d;
    RRTK_TRY(dev_info(&d));
    return plan_launch(kind, d_bits, W, H, d_plans, nplans, n, r_rewire, r_goal, d_samples, d_balls, d_pts, d_cost, d_parent,
                       d_stats, d_ell_c, threads, d->optin, d->sm_smem, (cudaStream_t)stream);
}

const char *rrtk_plan_kernel(int kind, int W, int H, int n, int threads)
{
    DevInfo *d;
    if (dev_info(&d) != RRTK_OK) return "";
    return plan_kernel_name(kind, W, H, n, threads, d->optin, d->sm_smem);
}

int rrtk_plan_footprint(int kind, int W, int H, int n, int threads, int *smem_bytes, int *blocks_per_sm)
{
    RRTK_TRY(check_grid_dims(W, H, 16384));
    DevInfo *d;
    RRTK_TRY(dev_info(&d));
    int rc = plan_footprint(kind, W, H, n, threads, d->optin, d->sm_smem, smem_bytes, blocks_per_sm);
    if (rc) set_error("plan with n=%d does not fit shared memory", n);
    return rc;
}

int rrtk_extract_paths(const int32_t *d_parent, const int64_t *d_stats, int nplans, int n, int cap, int32_t *d_path,
                       int32_t *d_len, void *stream)
{
    RRTK_REQUIRE(d_parent && d_stats && d_path && d_len && nplans >= 0 && n >= 1 && cap >= 1, "rrtk_extract_paths: bad argument");
    if (nplans == 0) return RRTK_OK;
    return paths_launch(d_parent, d_stats, nplans, n, cap, d_path, d_len, (cudaStream_t)stream);
}

int rrtk_extract_paths_xy(const int32_t *d_parent, const int16_t *d_pts, const double *d_cost, const int64_t *d_stats, int nplans,
                          int n, int cap, int32_t *d_path, int16_t *d_xy, int32_t *d_len, double *d_path_cost, void *stream)
{
    RRTK_REQUIRE(d_parent && d_pts && d_cost && d_stats && d_path && d_xy && d_len && d_path_cost && nplans >= 0 && n >= 1 && cap >= 1,
                 "rrtk_extract_paths_xy: bad argument");
    if (nplans == 0) return RRTK_OK;
    return paths_xy_launch(d_parent, d_pts, d_cost, d_stats, nplans, n, cap, d_path, d_xy, d_len, d_path_cost, (cudaStream_t)stream);
}

// ---- measured roofline denominators (csrc/peaks.cu) ---------------------------------------------------
int rrtk_peak_l2_read(const void *d_buf, size_t bytes, int passes, uint32_t *d_sink, int64_t *bytes_read, void *stream)
{
    RRTK_REQUIRE(d_buf && d_sink && bytes >= 4096 && passes >= 1, "rrtk_peak_l2_read: bad argument");
    DevInfo *d;
    RRTK_TRY(dev_info(&d));
    if (bytes_read) *bytes_read = (int64_t)(bytes / 16 * 16) * passes;
    return l2_read_launch(d_buf, bytes, passes, d->sms, d_sink, (cudaStream_t)stream);
}

int rrtk_peak_smem_read(int smem_bytes, int iters, uint32_t *d_sink, int64_t *bytes_read, void *stream)
{
    RRTK_REQUIRE(d_sink && iters >= 1, "rrtk_peak_smem_read: bad argument");
    DevInfo *d;
    RRTK_TRY(dev_info(&d));
    if (smem_bytes <= 0 || smem_bytes > d->optin) smem_bytes = d->optin;
    int words16 = smem_bytes / 16;
    words16 -= words16 % (1024 * 8);
    RRTK_REQUIRE(words16 > 0, "rrtk_peak_smem_read: need at least 128 KB of shared memory per block");
    if (bytes_read) *bytes_read = (int64_t)words16 * 16 * iters * d->sms;
    return smem_read_launch(words16 * 16, iters, d->sms, d_sink, (cudaStream_t)stream);
}

// ---- host-buffer context ---------------------------------------------------------------------------
int rrtk_create(rrtk_ctx **out)
{
    RRTK_REQUIRE(out, "rrtk_create: null pointer");
    *out = nullptr;
    if (rrtk_device_count() < 1) {
        set_error("no CUDA device visible: librrtk has no CPU fallback");
        return RRTK_ERR_NODEVICE;
    }
    rrtk_ctx *c = new rrtk_ctx();
    cudaError_t e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) { delete c; return cuda_fail(e, "cudaStreamCreate"); }
    *out = c;
    return RRTK_OK;
}

int rrtk_destroy(rrtk_ctx *c)
{
    if (!c) return RRTK_OK;
    DevBuf *all[] = {&c->og, &c->bits, &c->rowcum, &c->plans, &c->samples, &c->state, &c->balls, &c->pts,
                     &c->cost, &c->parent, &c->stats, &c->ell, &c->a, &c->b, &c->c, &c->d, &c->e,
                     &c->heads, &c->head_out, &c->elen, &c->scratch2, &c->dtable};
    for (DevBuf *b : all) b->release();
    for (PipeSlot &p : c->pipe) {
        DevBuf *pb[] = {&p.og, &p.bits, &p.rowcum, &p.plans, &p.samples, &p.state, &p.balls, &p.pts, &p.cost, &p.parent, &p.stats, &p.ell};
        for (DevBuf *b : pb) b->release();
        if (p.stream) cudaStreamDestroy(p.stream);
        if (p.ready) cudaEventDestroy(p.ready);
        if (p.planned) cudaEventDestroy(p.planned);
        if (p.done) cudaEventDestroy(p.done);
    }
    if (c->pin_nfree) cudaFreeHost(c->pin_nfree);
    if (c->pipe_prep) cudaStreamDestroy(c->pipe_prep);
    if (c->pipe_post) cudaStreamDestroy(c->pipe_post);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
    return RRTK_OK;
}

int rrtk_ctx_set_grids(rrtk_ctx *c, const uint8_t *h_og, int nworlds, int W, int H, int32_t *h_nfree)
{
    RRTK_REQUIRE(c && h_og && nworlds >= 1, "rrtk_ctx_set_grids: bad argument");
    RRTK_TRY(check_grid_dims(W, H, 16384));
    const size_t cells = (size_t)W * H;
    RRTK_TRY(c->og.reserve(cells * nworlds));
    RRTK_TRY(c->bits.reserve(grid_words(W, H) * 4 * nworlds));
    RRTK_TRY(c->rowcum.reserve((size_t)(W + 1) * 4 * nworlds));
    RRTK_CUDA(cudaMemcpyAsync(c->og.p, h_og, cells * nworlds, cudaMemcpyHostToDevice, c->stream));
    RRTK_TRY(pack_launch(c->og.as<uint8_t>(), nworlds, W, H, c->bits.as<uint32_t>(), c->stream));
    RRTK_TRY(free_rows_launch(c->bits.as<uint32_t>(), nworlds, W, H, c->rowcum.as<int32_t>(), c->stream));
    c->nworlds = 0;
    c->nfree.assign(nworlds, 0);
    RRTK_CUDA(cudaMemcpy2DAsync(c->nfree.data(), 4, c->rowcum.as<int32_t>() + W, (size_t)(W + 1) * 4, 4, nworlds,
                                cudaMemcpyDeviceToHost, c->stream));
    RRTK_CUDA(cudaStreamSynchronize(c->stream));
    if (h_nfree) memcpy(h_nfree, c->nfree.data(), (size_t)nworlds * 4);
    c->W = W; c->H = H; c->nworlds = nworlds;
    return RRTK_OK;
}

// seed mode draws free[choice(nfree)] (rrt.py:240): a world without a free cell has nothing to draw (numpy raises)
static int require_free_cells(const rrtk_ctx *c, const rrtk_plan_desc *h_plans, int nplans, const char *who)
{
    for (int p = 0; p < nplans; ++p) {
        const int w = h_plans[p].world;
        if (w >= 0 && w < c->nworlds && c->nfree[w] <= 0) {
            set_error("%s: world %d of plan %d has no free cell to sample", who, w, p);
            return RRTK_ERR_INVALID;
        }
    }
    return RRTK_OK;
}

int rrtk_ctx_inflate(rrtk_ctx *c, const uint8_t *h_og, int W, int H, int iterations, const int32_t *h_holes, int nout,
                     uint8_t *h_out)
{
    RRTK_REQUIRE(c && h_og && h_out && nout >= 1 && iterations >= 0, "rrtk_ctx_inflate: bad argument");
    RRTK_TRY(check_grid_dims(W, H, 16384));
    const size_t cells = (size_t)W * H, wb = grid_words(W, H) * 4;
    // scratch buffers of the context: a = source uint8 / result uint8, b = source bits, c = result bits, d = passes, e = holes
    RRTK_TRY(c->a.reserve(cells * nout));
    RRTK_TRY(c->b.reserve(wb));
    RRTK_TRY(c->c.reserve(wb * nout));
    RRTK_TRY(c->d.reserve(wb * 2));
    RRTK_TRY(c->e.reserve((size_t)nout * 12));
    RRTK_CUDA(cudaMemcpyAsync(c->a.p, h_og, cells, cudaMemcpyHostToDevice, c->stream));
    if (h_holes) RRTK_CUDA(cudaMemcpyAsync(c->e.p, h_holes, (size_t)nout * 12, cudaMemcpyHostToDevice, c->stream));
    RRTK_TRY(pack_launch(c->a.as<uint8_t>(), 1, W, H, c->b.as<uint32_t>(), c->stream));
    RRTK_TRY(inflate_launch(c->b.as<uint32_t>(), 1, W, H, iterations, h_holes ? c->e.as<int32_t>() : nullptr, nout,
                            c->c.as<uint32_t>(), c->d.as<uint32_t>(), c->stream));
    RRTK_TRY(unpack_launch(c->c.as<uint32_t>(), nout, W, H, c->a.as<uint8_t>(), c->stream));
    RRTK_CUDA(cudaMemcpyAsync(h_out, c->a.p, cells * nout, cudaMemcpyDeviceToHost, c->stream));
    RRTK_CUDA(cudaStreamSynchronize(c->stream));
    return RRTK_OK;
}

int rrtk_ctx_plan(rrtk_ctx *c, int kind, const rrtk_plan_desc *h_plans, int nplans, int n, double r_rewire, double r_goal,
                  const int16_t *h_samples, const uint64_t *h_state, const double *h_balls, int16_t *h_pts, double *h_cost,
                  int32_t *h_parent, int64_t *h_stats, double *h_ell_c)
{
    RRTK_REQUIRE(c && h_plans && h_pts && h_cost && h_parent && h_stats, "rrtk_ctx_plan: null pointer");
    RRTK_REQUIRE(c->nworlds > 0, "rrtk_ctx_plan: call rrtk_ctx_set_grids first");
    RRTK_REQUIRE((h_samples != nullptr) != (h_state != nullptr), "rrtk_ctx_plan: pass exactly one of h_samples / h_state");
    RRTK_REQUIRE(kind != RRTK_INFORMED || h_ell_c, "rrtk_ctx_plan: informed plans need h_ell_c");
    RRTK_REQUIRE(nplans >= 0 && n >= 1 && n <= 65534, "rrtk_ctx_plan: need nplans >= 0 and 1 <= n <= 65534");
    if (nplans == 0) return RRTK_OK;
    for (int p = 0; p < nplans; ++p) {
        const rrtk_plan_desc &d = h_plans[p];
        if (d.world < 0 || d.world >= c->nworlds || d.start_x < 0 || d.start_x >= c->W || d.goal_x < 0 || d.goal_x >= c->W ||
            d.start_y < 0 || d.start_y >= c->H || d.goal_y < 0 || d.goal_y >= c->H) {
            set_error("plan %d: world index or start/goal outside the grid", p);
            return RRTK_ERR_INVALID;
        }
    }
    if (h_samples) {
        const size_t total = (size_t)nplans * n;
        for (size_t i = 0; i < total; ++i) {
            const int x = h_samples[2 * i], y = h_samples[2 * i + 1];
            if (x < 0 || x >= c->W || y < 0 || y >= c->H) {
                set_error("sample %zu of plan %zu lies outside the grid", i % n, i / n);
                return RRTK_ERR_INVALID;
            }
        }
    }
    if (h_state) RRTK_TRY(require_free_cells(c, h_plans, nplans, "rrtk_ctx_plan"));
    const size_t rows = (size_t)nplans * (n + 1);
    cudaStream_t st = c->stream;
    RRTK_TRY(c->plans.reserve(sizeof(rrtk_plan_desc) * nplans));
    RRTK_TRY(c->samples.reserve((size_t)nplans * n * 4));
    RRTK_TRY(c->pts.reserve(rows * 4));
    RRTK_TRY(c->cost.reserve(rows * 8));
    RRTK_TRY(c->parent.reserve(rows * 4));
    RRTK_TRY(c->stats.reserve((size_t)nplans * RRTK_STAT_COUNT * 8));
    RRTK_CUDA(cudaMemcpyAsync(c->plans.p, h_plans, sizeof(rrtk_plan_desc) * nplans, cudaMemcpyHostToDevice, st));
    if (h_samples) {
        RRTK_CUDA(cudaMemcpyAsync(c->samples.p, h_samples, (size_t)nplans * n * 4, cudaMemcpyHostToDevice, st));
    } else {
        DevInfo *d;
        RRTK_TRY(dev_info(&d));
        RRTK_TRY(c->state.reserve((size_t)nplans * 32));
        RRTK_CUDA(cudaMemcpyAsync(c->state.p, h_state, (size_t)nplans * 32, cudaMemcpyHostToDevice, st));
        RRTK_TRY(sample_streams_launch(c->bits.as<uint32_t>(), c->rowcum.as<int32_t>(), c->W, c->H, c->plans.as<rrtk_plan_desc>(),
                                       nplans, c->state.as<uint64_t>(), n, c->samples.as<int16_t>(), d->optin, st));
    }
    if (kind == RRTK_INFORMED) {
        RRTK_TRY(c->ell.reserve(rows * 8));
        if (h_balls) {
            RRTK_TRY(c->balls.reserve((size_t)nplans * n * 16));
            RRTK_CUDA(cudaMemcpyAsync(c->balls.p, h_balls, (size_t)nplans * n * 16, cudaMemcpyHostToDevice, st));
        }
    }
    RRTK_TRY(rrtk_plan_batch(kind, c->bits.as<uint32_t>(), c->W, c->H, c->plans.as<rrtk_plan_desc>(), nplans, n, r_rewire, r_goal,
                             c->samples.as<int16_t>(), (kind == RRTK_INFORMED && h_balls) ? c->balls.as<double>() : nullptr,
                             c->pts.as<int16_t>(), c->cost.as<double>(),
                             c->parent.as<int32_t>(), c->stats.as<int64_t>(), c->ell.as<double>(), 0, st));
    RRTK_CUDA(cudaMemcpyAsync(h_pts, c->pts.p, rows * 4, cudaMemcpyDeviceToHost, st));
    RRTK_CUDA(cudaMemcpyAsync(h_cost, c->cost.p, rows * 8, cudaMemcpyDeviceToHost, st));
    RRTK_CUDA(cudaMemcpyAsync(h_parent, c->parent.p, rows * 4, cudaMemcpyDeviceToHost, st));
    RRTK_CUDA(cudaMemcpyAsync(h_stats, c->stats.p, (size_t)nplans * RRTK_STAT_COUNT * 8, cudaMemcpyDeviceToHost, st));
    if (kind == RRTK_INFORMED) RRTK_CUDA(cudaMemcpyAsync(h_ell_c, c->ell.p, rows * 8, cudaMemcpyDeviceToHost, st));
    RRTK_CUDA(cudaStreamSynchronize(st));
    return RRTK_OK;
}

// Upload, plan and download in chunks of plans on rotating streams, so that host<->device copies of
// one chunk overlap the kernels of its neighbours.  Plans must be ordered by world index.
// flags: RRTK_IN_BITS (h_grids = tiled bit grids, 1/8 of the bytes), RRTK_OUT_TREES, RRTK_OUT_PATHS (path records of
// path_cap entries per plan); statistics always come back.
// streams and events of one pipeline slot (and the two shared streams), created on first use; every pipelined call drains all of
// them before it returns, so the slot's buffers may be regrown right after this
static int pipe_slot_init(rrtk_ctx *c, PipeSlot &s)
{
    if (!c->pipe_prep) {
        int lo = 0, hi = 0;
        RRTK_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));                    // hi = numerically lowest = greatest priority
        RRTK_CUDA(cudaStreamCreateWithPriority(&c->pipe_prep, cudaStreamNonBlocking, hi));
        RRTK_CUDA(cudaStreamCreateWithPriority(&c->pipe_post, cudaStreamNonBlocking, hi));
    }
    if (!s.stream) {
        RRTK_CUDA(cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking));
        RRTK_CUDA(cudaEventCreateWithFlags(&s.ready, cudaEventDisableTiming));
        RRTK_CUDA(cudaEventCreateWithFlags(&s.planned, cudaEventDisableTiming));
        RRTK_CUDA(cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming));
    }
    return RRTK_OK;
}

static int pipe_nfree_reserve(rrtk_ctx *c, size_t nworlds)
{
    if (nworlds <= c->pin_nfree_cap) return RRTK_OK;
    if (c->pin_nfree) cudaFreeHost(c->pin_nfree);
    c->pin_nfree = nullptr; c->pin_nfree_cap = 0;
    RRTK_CUDA(cudaHostAlloc(reinterpret_cast<void **>(&c->pin_nfree), nworlds * sizeof(int32_t), cudaHostAllocDefault));
    c->pin_nfree_cap = nworlds;
    return RRTK_OK;
}

// seed mode draws free[choice(nfree)] (rrt.py:240): the results of a plan on a world without a free cell mean nothing
static int pipe_require_free_cells(const rrtk_ctx *c, const rrtk_plan_desc *h_plans, int nplans, const char *who)
{
    for (int p = 0; p < nplans; ++p)
        if (c->pin_nfree[h_plans[p].world] <= 0) {
            set_error("%s: world %d of plan %d has no free cell to sample", who, h_plans[p].world, p);
            return RRTK_ERR_INVALID;
        }
    return RRTK_OK;
}

// RRTK_SEED_BALLS: with start == goal the ellipse has no orientation (rotation_to_world_frame raises, rrt.py:601-613), which
// the reference meets only once the plan reaches the ellipse phase, i.e. once it has a first solution vertex
static int pipe_require_rotations(const rrtk_plan_desc *h_plans, const int64_t *h_stats, int nplans, int first_col, const char *who)
{
    for (int p = 0; p < nplans; ++p) {
        const double *r = h_plans[p].rot;
        if (h_stats[(size_t)p * RRTK_STAT_COUNT + first_col] >= 0 &&
            !(std::isfinite(r[0]) && std::isfinite(r[1]) && std::isfinite(r[2]) && std::isfinite(r[3]))) {
            set_error("%s: plan %d reaches the ellipse phase but its rotation is not finite (start == goal)", who, p);
            return RRTK_ERR_INVALID;
        }
    }
    return RRTK_OK;
}

static void pipe_drain(rrtk_ctx *c, int *status)
{
    auto sync = [&](cudaStream_t st) {
        if (!st) return;
        const cudaError_t e = cudaStreamSynchronize(st);
        if (e != cudaSuccess && *status == RRTK_OK) *status = cuda_fail(e, "cudaStreamSynchronize");
    };
    sync(c->pipe_prep);
    for (PipeSlot &s : c->pipe) sync(s.stream);
    sync(c->pipe_post);
}

int rrtk_ctx_plan_worlds2(rrtk_ctx *c, int kind, const void *h_grids, int nworlds, int W, int H, const rrtk_plan_desc *h_plans,
                          int nplans, int n, double r_rewire, double r_goal, const int16_t *h_samples, const uint64_t *h_state,
                          const double *h_balls, int flags, int path_cap, int16_t *h_pts, double *h_cost, int32_t *h_parent,
                          int64_t *h_stats, double *h_ell_c, int32_t *h_path, int16_t *h_xy, int32_t *h_len, double *h_path_cost,
                          int chunk_plans)
{
    const bool in_bits = flags & RRTK_IN_BITS, out_trees = flags & RRTK_OUT_TREES, out_paths = flags & RRTK_OUT_PATHS;
    const bool seed_balls = flags & RRTK_SEED_BALLS;
    RRTK_REQUIRE(!seed_balls || h_state, "rrtk_ctx_plan_worlds2: RRTK_SEED_BALLS needs seed mode (h_state)");
    RRTK_REQUIRE(!seed_balls || kind == RRTK_INFORMED, "rrtk_ctx_plan_worlds2: RRTK_SEED_BALLS needs kind RRTK_INFORMED");
    RRTK_REQUIRE(!seed_balls || !h_balls, "rrtk_ctx_plan_worlds2: RRTK_SEED_BALLS draws the unit-disc stream itself (pass h_balls = NULL)");
    RRTK_REQUIRE(c && h_grids && h_plans && h_stats, "rrtk_ctx_plan_worlds2: null pointer");
    RRTK_REQUIRE(!out_trees || (h_pts && h_cost && h_parent), "rrtk_ctx_plan_worlds2: RRTK_OUT_TREES needs h_pts, h_cost, h_parent");
    RRTK_REQUIRE(!out_paths || (h_path && h_xy && h_len && h_path_cost && path_cap >= 1),
                 "rrtk_ctx_plan_worlds2: RRTK_OUT_PATHS needs h_path, h_xy, h_len, h_path_cost and path_cap >= 1");
    RRTK_REQUIRE((h_samples != nullptr) != (h_state != nullptr), "rrtk_ctx_plan_worlds2: pass exactly one of h_samples / h_state");
    RRTK_REQUIRE(kind != RRTK_INFORMED || !out_trees || h_ell_c, "rrtk_ctx_plan_worlds2: informed trees need h_ell_c");
    RRTK_REQUIRE(nworlds >= 1 && nplans >= 0 && n >= 1 && n <= 65534, "rrtk_ctx_plan_worlds2: need nworlds >= 1, nplans >= 0, 1 <= n <= 65534");
    RRTK_TRY(check_grid_dims(W, H, 16384));
    if (nplans == 0) return RRTK_OK;
    bool ramp = false;
    if (chunk_plans <= 0) {
        // Chunks of two plan blocks per SM (a fraction of a wave): the next chunks' uploads, packing and sampler kernel
        // need free SM resources to overlap the running plan blocks, and a chunk that fills every SM leaves none until
        // its first blocks retire.  Measured on B200, cfg3, 4096 plans (scripts/e2e_breakdown.py): 222..740 plans per
        // chunk 61.6-64 ms, 1036 (one wave) 75 ms, unpipelined 82 ms.
        DevInfo *di;
        RRTK_TRY(dev_info(&di));
        int smem = 0, per_sm = 0;
        chunk_plans = 2 * di->sms;
        // with packed grids in and no trees out the copies are small and the per-chunk fixed costs dominate: four blocks per SM
        // (measured, same workload: 296 / 592 / 1036 / 4096 plans per chunk -> 75.1 / 79.2 / 78.6 / 77.8 k plans/s)
        if (in_bits && !out_trees) chunk_plans = 4 * di->sms;
        if (plan_footprint(kind, W, H, n, 0, di->optin, di->sm_smem, &smem, &per_sm) == RRTK_OK && per_sm > 0 && per_sm < 2)
            chunk_plans = di->sms * per_sm;
        ramp = true;
    }
    for (int p = 0; p < nplans; ++p) {
        const rrtk_plan_desc &d = h_plans[p];
        if (d.world < 0 || d.world >= nworlds || d.start_x < 0 || d.start_x >= W || d.goal_x < 0 || d.goal_x >= W ||
            d.start_y < 0 || d.start_y >= H || d.goal_y < 0 || d.goal_y >= H) {
            set_error("plan %d: world index or start/goal outside the grid", p);
            return RRTK_ERR_INVALID;
        }
        if (p && d.world < h_plans[p - 1].world) {
            set_error("rrtk_ctx_plan_worlds: plans must be ordered by world index (plan %d)", p);
            return RRTK_ERR_INVALID;
        }
    }
    if (h_samples) {
        const size_t total = (size_t)nplans * n;
        for (size_t i = 0; i < total; ++i) {
            const int x = h_samples[2 * i], y = h_samples[2 * i + 1];
            if (x < 0 || x >= W || y < 0 || y >= H) {
                set_error("sample %zu of plan %zu lies outside the grid", i % n, i / n);
                return RRTK_ERR_INVALID;
            }
        }
    }
    DevInfo *di;
    RRTK_TRY(dev_info(&di));
    const size_t cells = (size_t)W * H, words = grid_words(W, H), rows1 = (size_t)n + 1;
    const size_t grid_bytes = in_bits ? words * 4 : cells;
    // chunk list, then every slot sized once for the largest chunk (growing a buffer later would free it under the pipeline)
    std::vector<int> starts;
    {
        int sz = ramp ? (di->sms < chunk_plans ? di->sms : chunk_plans) : chunk_plans;
        for (int p0 = 0; p0 < nplans; p0 += sz, sz = (2 * sz < chunk_plans) ? 2 * sz : chunk_plans) {
            starts.push_back(p0);
            if (p0 + sz >= nplans) break;
        }
        starts.push_back(nplans);
    }
    size_t max_m = 0, max_nw = 0;
    for (size_t k = 0; k + 1 < starts.size(); ++k) {
        const size_t m = (size_t)(starts[k + 1] - starts[k]);
        const size_t nw = (size_t)(h_plans[starts[k + 1] - 1].world - h_plans[starts[k]].world + 1);
        max_m = m > max_m ? m : max_m;
        max_nw = nw > max_nw ? nw : max_nw;
    }
    // Everything that can fail on the host side happens before the first copy is enqueued; from then on an error is
    // recorded, the loop stops, and every stream is drained before returning, so that no copy is still writing into the
    // caller's buffers when the call comes back.
    int status = RRTK_OK;
    auto cuda_ok = [&](cudaError_t e, const char *what) {
        if (e != cudaSuccess && status == RRTK_OK) status = cuda_fail(e, what);
        return e == cudaSuccess;
    };
    auto rrtk_ok = [&](int rc) {
        if (rc != RRTK_OK && status == RRTK_OK) status = rc;
        return rc == RRTK_OK;
    };
    if (h_state) RRTK_TRY(pipe_nfree_reserve(c, (size_t)nworlds));
    const size_t nslots = starts.size() - 1 < (size_t)kPipeSlots ? starts.size() - 1 : (size_t)kPipeSlots;
    for (size_t k = 0; k < nslots && status == RRTK_OK; ++k) {
        PipeSlot &s = c->pipe[k];
        if (!rrtk_ok(pipe_slot_init(c, s))) break;
        bool ok = rrtk_ok(s.bits.reserve(words * 4 * max_nw)) && rrtk_ok(s.rowcum.reserve((size_t)(W + 1) * 4 * max_nw)) &&
                  rrtk_ok(s.plans.reserve(sizeof(rrtk_plan_desc) * max_m)) && rrtk_ok(s.samples.reserve(max_m * n * 4)) &&
                  rrtk_ok(s.state.reserve(max_m * 32)) && rrtk_ok(s.pts.reserve(rows1 * max_m * 4)) &&
                  rrtk_ok(s.cost.reserve(rows1 * max_m * 8)) && rrtk_ok(s.parent.reserve(rows1 * max_m * 4)) &&
                  rrtk_ok(s.stats.reserve(max_m * RRTK_STAT_COUNT * 8));
        if (ok && !in_bits) ok = rrtk_ok(s.og.reserve(cells * max_nw));
        if (ok && kind == RRTK_INFORMED)
            ok = rrtk_ok(s.ell.reserve(rows1 * max_m * 8)) && ((!h_balls && !seed_balls) || rrtk_ok(s.balls.reserve(max_m * n * 16)));
        if (ok && out_paths)
            ok = rrtk_ok(s.path.reserve(max_m * path_cap * 4)) && rrtk_ok(s.xy.reserve(max_m * path_cap * 4)) &&
                 rrtk_ok(s.len.reserve(max_m * 4)) && rrtk_ok(s.pcost.reserve(max_m * 8));
    }
    // RRTK_PIPE_TRACE=1 (diagnosis): device-side time stamps of every chunk's stages, printed to stderr after the call
    const bool trace = getenv("RRTK_PIPE_TRACE") != nullptr;
    std::vector<cudaEvent_t> tev;
    auto stamp = [&](cudaStream_t on) {
        if (!trace) return;
        cudaEvent_t e = nullptr;
        cudaEventCreate(&e);
        cudaEventRecord(e, on);
        tev.push_back(e);
    };
    const auto host_t0 = std::chrono::steady_clock::now();
    std::vector<double> host_ms;
    for (size_t ci = 0; ci + 1 < starts.size() && status == RRTK_OK; ++ci) {
        const int p0 = starts[ci], m = starts[ci + 1] - starts[ci];
        PipeSlot &s = c->pipe[ci % kPipeSlots];
        cudaStream_t st = c->pipe_prep;                                           // preparation first (see PipeSlot), then the plan stream
        if (trace) host_ms.push_back(std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - host_t0).count());
        stamp(st);                                                                // [0] preparation of the chunk begins
        if (ci >= (size_t)kPipeSlots && !cuda_ok(cudaStreamWaitEvent(st, s.done, 0), "cudaStreamWaitEvent")) break;   // the slot's last chunk still reads these buffers
        const int w0 = h_plans[p0].world, w1 = h_plans[p0 + m - 1].world, nw = w1 - w0 + 1;
        const uint8_t *src = static_cast<const uint8_t *>(h_grids) + grid_bytes * w0;
        if (in_bits) {
            if (!cuda_ok(cudaMemcpyAsync(s.bits.p, src, grid_bytes * nw, cudaMemcpyHostToDevice, st), "cudaMemcpyAsync(bits)")) break;
        } else {
            if (!cuda_ok(cudaMemcpyAsync(s.og.p, src, grid_bytes * nw, cudaMemcpyHostToDevice, st), "cudaMemcpyAsync(og)")) break;
            if (!rrtk_ok(pack_launch(s.og.as<uint8_t>(), nw, W, H, s.bits.as<uint32_t>(), st))) break;
        }
        if (!rrtk_ok(free_rows_launch(s.bits.as<uint32_t>(), nw, W, H, s.rowcum.as<int32_t>(), st))) break;
        if (h_state && !cuda_ok(cudaMemcpy2DAsync(c->pin_nfree + w0, 4, s.rowcum.as<int32_t>() + W, (size_t)(W + 1) * 4, 4, nw, cudaMemcpyDeviceToHost, st),
                                "cudaMemcpy2DAsync(nfree)")) break;
        s.desc.assign(h_plans + p0, h_plans + p0 + m);
        for (rrtk_plan_desc &d : s.desc) d.world -= w0;
        if (!cuda_ok(cudaMemcpyAsync(s.plans.p, s.desc.data(), sizeof(rrtk_plan_desc) * m, cudaMemcpyHostToDevice, st), "cudaMemcpyAsync(plans)")) break;
        if (h_samples) {
            if (!cuda_ok(cudaMemcpyAsync(s.samples.p, h_samples + (size_t)p0 * n * 2, (size_t)m * n * 4, cudaMemcpyHostToDevice, st), "cudaMemcpyAsync(samples)")) break;
        } else {
            if (!cuda_ok(cudaMemcpyAsync(s.state.p, h_state + (size_t)p0 * 4, (size_t)m * 32, cudaMemcpyHostToDevice, st), "cudaMemcpyAsync(state)")) break;
            if (!rrtk_ok(sample_streams_launch(s.bits.as<uint32_t>(), s.rowcum.as<int32_t>(), W, H, s.plans.as<rrtk_plan_desc>(), m,
                                               s.state.as<uint64_t>(), n, s.samples.as<int16_t>(), di->optin, st))) break;
        }
        if (kind == RRTK_INFORMED && h_balls &&
            !cuda_ok(cudaMemcpyAsync(s.balls.p, h_balls + (size_t)p0 * n * 2, (size_t)m * n * 16, cudaMemcpyHostToDevice, st), "cudaMemcpyAsync(balls)")) break;
        if (!cuda_ok(cudaEventRecord(s.ready, st), "cudaEventRecord")) break;
        stamp(st);                                                                // [1] inputs ready
        st = s.stream;
        if (!cuda_ok(cudaStreamWaitEvent(st, s.ready, 0), "cudaStreamWaitEvent")) break;
        stamp(st);                                                                // [2] plan stream free and inputs ready
        if (seed_balls) {
            // probe (stops at the first solution vertex), then the unit-disc stream from the generator past that iteration
            if (!rrtk_ok(rrtk_plan_batch(kind, s.bits.as<uint32_t>(), W, H, s.plans.as<rrtk_plan_desc>(), m, n, r_rewire, r_goal,
                                         s.samples.as<int16_t>(), nullptr, s.pts.as<int16_t>(), s.cost.as<double>(), s.parent.as<int32_t>(),
                                         s.stats.as<int64_t>(), s.ell.as<double>(), 0, st))) break;
            if (!rrtk_ok(ball_streams_launch(s.rowcum.as<int32_t>(), W, s.plans.as<rrtk_plan_desc>(), m, n, s.state.as<uint64_t>(), nullptr,
                                             s.stats.as<int64_t>() + RRTK_STAT_FIRST_SOL_ITER, RRTK_STAT_COUNT, s.balls.as<double>(), nullptr,
                                             nullptr, st))) break;
        }
        if (!rrtk_ok(rrtk_plan_batch(kind, s.bits.as<uint32_t>(), W, H, s.plans.as<rrtk_plan_desc>(), m, n, r_rewire, r_goal,
                                     s.samples.as<int16_t>(), (kind == RRTK_INFORMED && (h_balls || seed_balls)) ? s.balls.as<double>() : nullptr,
                                     s.pts.as<int16_t>(), s.cost.as<double>(), s.parent.as<int32_t>(), s.stats.as<int64_t>(),
                                     s.ell.as<double>(), 0, st))) break;
        stamp(st);                                                                // [3] plan kernel done
        if (!cuda_ok(cudaEventRecord(s.planned, st), "cudaEventRecord")) break;
        st = c->pipe_post;                                                        // outputs: extraction and downloads, high priority
        if (!cuda_ok(cudaStreamWaitEvent(st, s.planned, 0), "cudaStreamWaitEvent")) break;
        bool ok = true;
        if (out_paths) {
            ok = rrtk_ok(paths_xy_launch(s.parent.as<int32_t>(), s.pts.as<int16_t>(), s.cost.as<double>(), s.stats.as<int64_t>(), m, n, path_cap,
                                         s.path.as<int32_t>(), s.xy.as<int16_t>(), s.len.as<int32_t>(), s.pcost.as<double>(), st)) &&
                 cuda_ok(cudaMemcpyAsync(h_path + (size_t)p0 * path_cap, s.path.p, (size_t)m * path_cap * 4, cudaMemcpyDeviceToHost, st), "cudaMemcpyAsync(path)") &&
                 cuda_ok(cudaMemcpyAsync(h_xy + (size_t)p0 * path_cap * 2, s.xy.p, (size_t)m * path_cap * 4, cudaMemcpyDeviceToHost, st), "cudaMemcpyAsync(xy)") &&
                 cuda_ok(cudaMemcpyAsync(h_len + p0, s.len.p, (size_t)m * 4, cudaMemcpyDeviceToHost, st), "cudaMemcpyAsync(len)") &&
                 cuda_ok(cudaMemcpyAsync(h_path_cost + p0, s.pcost.p, (size_t)m * 8, cudaMemcpyDeviceToHost, st), "cudaMemcpyAsync(path_cost)");
        }
        if (ok && out_trees) {
            ok = cuda_ok(cudaMemcpyAsync(h_pts + (size_t)p0 * rows1 * 2, s.pts.p, rows1 * m * 4, cudaMemcpyDeviceToHost, st), "cudaMemcpyAsync(pts)") &&
                 cuda_ok(cudaMemcpyAsync(h_cost + (size_t)p0 * rows1, s.cost.p, rows1 * m * 8, cudaMemcpyDeviceToHost, st), "cudaMemcpyAsync(cost)") &&
                 cuda_ok(cudaMemcpyAsync(h_parent + (size_t)p0 * rows1, s.parent.p, rows1 * m * 4, cudaMemcpyDeviceToHost, st), "cudaMemcpyAsync(parent)");
            if (ok && kind == RRTK_INFORMED)
                ok = cuda_ok(cudaMemcpyAsync(h_ell_c + (size_t)p0 * rows1, s.ell.p, rows1 * m * 8, cudaMemcpyDeviceToHost, st), "cudaMemcpyAsync(ell)");
        }
        if (ok) cuda_ok(cudaMemcpyAsync(h_stats + (size_t)p0 * RRTK_STAT_COUNT, s.stats.p, (size_t)m * RRTK_STAT_COUNT * 8, cudaMemcpyDeviceToHost, st), "cudaMemcpyAsync(stats)");
        cuda_ok(cudaEventRecord(s.done, st), "cudaEventRecord");
        stamp(st);                                                                // [4] results on the host
    }
    pipe_drain(c, &status);
    if (trace && status == RRTK_OK && tev.size() == 5 * (starts.size() - 1)) {
        const double host_end = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - host_t0).count();
        fprintf(stderr, "rrtk pipe trace (ms after the first chunk's preparation began; host = when the host enqueued the chunk; call returned at host %.2f)\n", host_end);
        for (size_t ci = 0; ci + 1 < starts.size(); ++ci) {
            float t[5];
            for (int k = 0; k < 5; ++k) cudaEventElapsedTime(&t[k], tev[0], tev[5 * ci + k]);
            fprintf(stderr, "  chunk %2zu plans %5d..%5d host %6.2f | prep %6.2f ready %6.2f | plan start %6.2f end %6.2f | out %6.2f\n", ci, starts[ci],
                    starts[ci + 1], host_ms[ci], t[0], t[1], t[2], t[3], t[4]);
        }
    }
    for (cudaEvent_t e : tev) cudaEventDestroy(e);
    if (status == RRTK_OK && h_state) status = pipe_require_free_cells(c, h_plans, nplans, "rrtk_ctx_plan_worlds2");
    if (status == RRTK_OK && seed_balls) status = pipe_require_rotations(h_plans, h_stats, nplans, RRTK_STAT_FIRST_SOL_ITER, "rrtk_ctx_plan_worlds2");
    return status;
}

// the round-1 form: uint8 grids in, every tree out
int rrtk_ctx_plan_worlds(rrtk_ctx *c, int kind, const uint8_t *h_og, int nworlds, int W, int H, const rrtk_plan_desc *h_plans,
                         int nplans, int n, double r_rewire, double r_goal, const int16_t *h_samples, const uint64_t *h_state,
                         const double *h_balls, int16_t *h_pts, double *h_cost, int32_t *h_parent, int64_t *h_stats,
                         double *h_ell_c, int chunk_plans)
{
    RRTK_REQUIRE(c && h_og && h_plans && h_pts && h_cost && h_parent && h_stats, "rrtk_ctx_plan_worlds: null pointer");
    RRTK_REQUIRE(kind != RRTK_INFORMED || h_ell_c, "rrtk_ctx_plan_worlds: informed plans need h_ell_c");
    return rrtk_ctx_plan_worlds2(c, kind, h_og, nworlds, W, H, h_plans, nplans, n, r_rewire, r_goal, h_samples, h_state, h_balls,
                                 RRTK_OUT_TREES, 0, h_pts, h_cost, h_parent, h_stats, h_ell_c, nullptr, nullptr, nullptr, nullptr, chunk_plans);
}

// np.random.default_rng(seed) -> PCG64 start state, on the host (rrt.py:85).  numpy's published seeding path: SeedSequence
// (numpy/random/bit_generator.pyx: hashmix / mix over a 4-word pool, generate_state(4, uint64)) feeds
// pcg_setseq_128_srandom_r (numpy/random/src/pcg64/pcg64.h).  h_state: {state_hi, state_lo, inc_hi, inc_lo} per seed.
int rrtk_seed_states(const uint64_t *h_seeds, int nseeds, uint64_t *h_state)
{
    RRTK_REQUIRE(h_seeds && h_state && nseeds >= 0, "rrtk_seed_states: null pointer or negative count");
    typedef unsigned __int128 u128;
    const u128 mult = ((u128)0x2360ED051FC65DA4ull << 64) | 0x4385DF649FCCF645ull;
    for (int i = 0; i < nseeds; ++i) {
        const uint32_t ent[4] = {(uint32_t)h_seeds[i], (uint32_t)(h_seeds[i] >> 32), 0u, 0u};
        uint32_t hc = 0x43B0D7E5u, pool[4];
        auto hashmix = [&](uint32_t v) { v ^= hc; hc *= 0x931E8875u; v *= hc; return v ^ (v >> 16); };
        auto mix = [](uint32_t x, uint32_t y) { const uint32_t r = 0xCA01F9DDu * x - 0x4973F715u * y; return r ^ (r >> 16); };
        for (int k = 0; k < 4; ++k) pool[k] = hashmix(ent[k]);
        for (int src = 0; src < 4; ++src)
            for (int dst = 0; dst < 4; ++dst)
                if (src != dst) pool[dst] = mix(pool[dst], hashmix(pool[src]));
        uint32_t hb = 0x8B51F9DDu, w32[8];
        for (int k = 0; k < 8; ++k) { uint32_t v = pool[k & 3] ^ hb; hb *= 0x58F38DEDu; v *= hb; w32[k] = v ^ (v >> 16); }
        uint64_t w[4];
        for (int k = 0; k < 4; ++k) w[k] = (uint64_t)w32[2 * k] | ((uint64_t)w32[2 * k + 1] << 32);
        const u128 initstate = ((u128)w[0] << 64) | w[1], initseq = ((u128)w[2] << 64) | w[3];
        const u128 inc = (initseq << 1) | 1u;
        u128 st = 0;
        st = st * mult + inc;
        st += initstate;
        st = st * mult + inc;
        uint64_t *o = h_state + 4 * (size_t)i;
        o[0] = (uint64_t)(st >> 64); o[1] = (uint64_t)st; o[2] = (uint64_t)(inc >> 64); o[3] = (uint64_t)inc;
    }
    return RRTK_OK;
}

// K0 on the host (include/rrtk.h: the tiled bit layout), for callers that keep their worlds packed
int rrtk_pack_grid_host(const uint8_t *h_og, int nworlds, int W, int H, uint32_t *h_bits)
{
    RRTK_REQUIRE(h_og && h_bits && nworlds >= 0, "rrtk_pack_grid_host: null pointer or negative count");
    RRTK_TRY(check_grid_dims(W, H, 32768));
    const int TX = tiles_x(W), TY = tiles_y(H);
    const size_t words = grid_words(W, H), cells = (size_t)W * H;
    for (int w = 0; w < nworlds; ++w) {
        const uint8_t *og = h_og + cells * w;
        uint32_t *bits = h_bits + words * w;
        for (int tx = 0; tx < TX; ++tx)
            for (int ty = 0; ty < TY; ++ty)
                for (int xl = 0; xl < 32; ++xl) {
                    const int x = tx * 32 + xl;
                    uint32_t word = 0xffffffffu;                                 // cells outside the grid count as occupied
                    if (x < W) {
                        word = 0u;
                        for (int b = 0; b < 32; ++b) {
                            const int y = ty * 32 + b;
                            if (y >= H || og[(size_t)x * H + y] != 0) word |= 1u << b;
                        }
                    }
                    bits[(((size_t)tx * TY + ty) << 5) | xl] = word;
                }
    }
    return RRTK_OK;
}

int rrtk_ctx_samples(rrtk_ctx *c, const rrtk_plan_desc *h_plans, int nplans, int n, const uint64_t *h_state, int16_t *h_samples)
{
    RRTK_REQUIRE(c && h_plans && h_state && h_samples && nplans >= 1 && n >= 1, "rrtk_ctx_samples: bad argument");
    RRTK_REQUIRE(c->nworlds > 0, "rrtk_ctx_samples: call rrtk_ctx_set_grids first");
    for (int p = 0; p < nplans; ++p) RRTK_REQUIRE(h_plans[p].world >= 0 && h_plans[p].world < c->nworlds, "rrtk_ctx_samples: bad world index");
    RRTK_TRY(require_free_cells(c, h_plans, nplans, "rrtk_ctx_samples"));
    DevInfo *d;
    RRTK_TRY(dev_info(&d));
    cudaStream_t st = c->stream;
    RRTK_TRY(c->plans.reserve(sizeof(rrtk_plan_desc) * nplans));
    RRTK_TRY(c->samples.reserve((size_t)nplans * n * 4));
    RRTK_TRY(c->state.reserve((size_t)nplans * 32));
    RRTK_CUDA(cudaMemcpyAsync(c->plans.p, h_plans, sizeof(rrtk_plan_desc) * nplans, cudaMemcpyHostToDevice, st));
    RRTK_CUDA(cudaMemcpyAsync(c->state.p, h_state, (size_t)nplans * 32, cudaMemcpyHostToDevice, st));
    RRTK_TRY(sample_streams_launch(c->bits.as<uint32_t>(), c->rowcum.as<int32_t>(), c->W, c->H, c->plans.as<rrtk_plan_desc>(), nplans,
                                   c->state.as<uint64_t>(), n, c->samples.as<int16_t>(), d->optin, st));
    RRTK_CUDA(cudaMemcpyAsync(h_samples, c->samples.p, (size_t)nplans * n * 4, cudaMemcpyDeviceToHost, st));
    RRTK_CUDA(cudaStreamSynchronize(st));
    return RRTK_OK;
}

int rrtk_ctx_collision(rrtk_ctx *c, int world, const int32_t *h_segs, int64_t nseg, uint8_t *h_free, int32_t *h_cells)
{
    RRTK_REQUIRE(c && nseg >= 0 && (nseg == 0 || (h_segs && h_free)), "rrtk_ctx_collision: bad argument");
    RRTK_REQUIRE(c->nworlds > 0 && world >= 0 && world < c->nworlds, "rrtk_ctx_collision: no such world (call rrtk_ctx_set_grids)");
    if (nseg == 0) return RRTK_OK;
    for (int64_t s = 0; s < nseg; ++s) {
        const int32_t *e = h_segs + 4 * s;
        if (e[0] < 0 || e[0] >= c->W || e[2] < 0 || e[2] >= c->W || e[1] < 0 || e[1] >= c->H || e[3] < 0 || e[3] >= c->H) {
            set_error("segment %lld has an endpoint outside the (%d, %d) grid", (long long)s, c->W, c->H);
            return RRTK_ERR_INVALID;
        }
    }
    cudaStream_t st = c->stream;
    RRTK_TRY(c->a.reserve((size_t)nseg * 16));
    RRTK_TRY(c->b.reserve((size_t)nseg));
    RRTK_TRY(c->c.reserve((size_t)nseg * 4));
    RRTK_CUDA(cudaMemcpyAsync(c->a.p, h_segs, (size_t)nseg * 16, cudaMemcpyHostToDevice, st));
    const uint32_t *bits = c->bits.as<uint32_t>() + (size_t)world * grid_words(c->W, c->H);
    RRTK_TRY(rrtk_collision_segments(bits, c->W, c->H, c->a.as<int32_t>(), nullptr, nseg, c->b.as<uint8_t>(), c->c.as<int32_t>(), st));
    RRTK_CUDA(cudaMemcpyAsync(h_free, c->b.p, (size_t)nseg, cudaMemcpyDeviceToHost, st));
    if (h_cells) RRTK_CUDA(cudaMemcpyAsync(h_cells, c->c.p, (size_t)nseg * 4, cudaMemcpyDeviceToHost, st));
    RRTK_CUDA(cudaStreamSynchronize(st));
    return RRTK_OK;
}

int rrtk_ctx_nearest(rrtk_ctx *c, const int32_t *h_pts, int npts, const int32_t *h_queries, int nq, int32_t *h_idx, int64_t *h_d2)
{
    RRTK_REQUIRE(c && npts >= 1 && nq >= 1 && h_pts && h_queries && h_idx, "rrtk_ctx_nearest: bad argument");
    cudaStream_t st = c->stream;
    RRTK_TRY(c->a.reserve((size_t)npts * 8));
    RRTK_TRY(c->b.reserve((size_t)nq * 8));
    RRTK_TRY(c->c.reserve((size_t)nq * 4));
    RRTK_TRY(c->d.reserve((size_t)nq * 8));
    RRTK_CUDA(cudaMemcpyAsync(c->a.p, h_pts, (size_t)npts * 8, cudaMemcpyHostToDevice, st));
    RRTK_CUDA(cudaMemcpyAsync(c->b.p, h_queries, (size_t)nq * 8, cudaMemcpyHostToDevice, st));
    RRTK_TRY(nearest_launch(c->a.as<int32_t>(), npts, c->b.as<int32_t>(), nullptr, nq, c->c.as<int32_t>(), c->d.as<int64_t>(), st));
    RRTK_CUDA(cudaMemcpyAsync(h_idx, c->c.p, (size_t)nq * 4, cudaMemcpyDeviceToHost, st));
    if (h_d2) RRTK_CUDA(cudaMemcpyAsync(h_d2, c->d.p, (size_t)nq * 8, cudaMemcpyDeviceToHost, st));
    RRTK_CUDA(cudaStreamSynchronize(st));
    return RRTK_OK;
}
int rrtk_ctx_nearest_f64(rrtk_ctx *c, const double *h_pts, int npts, const double *h_queries, int nq, int32_t *h_idx, double *h_dist)
{
    RRTK_REQUIRE(c && npts >= 1 && nq >= 1 && h_pts && h_queries && h_idx, "rrtk_ctx_nearest_f64: bad argument");
    cudaStream_t st = c->stream;
    RRTK_TRY(c->a.reserve((size_t)npts * 16));
    RRTK_TRY(c->b.reserve((size_t)nq * 16));
    RRTK_TRY(c->c.reserve((size_t)nq * 4));
    RRTK_TRY(c->d.reserve((size_t)nq * 8));
    RRTK_CUDA(cudaMemcpyAsync(c->a.p, h_pts, (size_t)npts * 16, cudaMemcpyHostToDevice, st));
    RRTK_CUDA(cudaMemcpyAsync(c->b.p, h_queries, (size_t)nq * 16, cudaMemcpyHostToDevice, st));
    RRTK_TRY(nearest_launch_f64(c->a.as<double>(), npts, c->b.as<double>(), nullptr, nq, c->c.as<int32_t>(), c->d.as<double>(), st));
    RRTK_CUDA(cudaMemcpyAsync(h_idx, c->c.p, (size_t)nq * 4, cudaMemcpyDeviceToHost, st));
    if (h_dist) RRTK_CUDA(cudaMemcpyAsync(h_dist, c->d.p, (size_t)nq * 8, cudaMemcpyDeviceToHost, st));
    RRTK_CUDA(cudaStreamSynchronize(st));
    return RRTK_OK;
}

int rrtk_ctx_within(rrtk_ctx *c, const int32_t *h_pts, int npts, const int32_t *h_queries, int nq, double r, int cap,
                    int32_t *h_out, int32_t *h_len)
{
    RRTK_REQUIRE(c && npts >= 1 && nq >= 1 && cap >= 1 && h_pts && h_queries && h_out && h_len, "rrtk_ctx_within: bad argument");
    cudaStream_t st = c->stream;
    RRTK_TRY(c->a.reserve((size_t)npts * 8));
    RRTK_TRY(c->b.reserve((size_t)nq * 8));
    RRTK_TRY(c->c.reserve((size_t)nq * cap * 4));
    RRTK_TRY(c->d.reserve((size_t)nq * 4));
    RRTK_CUDA(cudaMemcpyAsync(c->a.p, h_pts, (size_t)npts * 8, cudaMemcpyHostToDevice, st));
    RRTK_CUDA(cudaMemcpyAsync(c->b.p, h_queries, (size_t)nq * 8, cudaMemcpyHostToDevice, st));
    RRTK_TRY(within_launch(c->a.as<int32_t>(), npts, c->b.as<int32_t>(), nullptr, nq, r, cap, c->c.as<int32_t>(), c->d.as<int32_t>(), st));
    RRTK_CUDA(cudaMemcpyAsync(h_out, c->c.p, (size_t)nq * cap * 4, cudaMemcpyDeviceToHost, st));
    RRTK_CUDA(cudaMemcpyAsync(h_len, c->d.p, (size_t)nq * 4, cudaMemcpyDeviceToHost, st));
    RRTK_CUDA(cudaStreamSynchronize(st));
    return RRTK_OK;
}
int rrtk_ctx_within_f64(rrtk_ctx *c, const double *h_pts, int npts, const double *h_queries, int nq, double r, int cap,
                        int32_t *h_out, int32_t *h_len)
{
    RRTK_REQUIRE(c && npts >= 1 && nq >= 1 && cap >= 1 && h_pts && h_queries && h_out && h_len, "rrtk_ctx_within_f64: bad argument");
    cudaStream_t st = c->stream;
    RRTK_TRY(c->a.reserve((size_t)npts * 16));
    RRTK_TRY(c->b.reserve((size_t)nq * 16));
    RRTK_TRY(c->c.reserve((size_t)nq * cap * 4));
    RRTK_TRY(c->d.reserve((size_t)nq * 4));
    RRTK_CUDA(cudaMemcpyAsync(c->a.p, h_pts, (size_t)npts * 16, cudaMemcpyHostToDevice, st));
    RRTK_CUDA(cudaMemcpyAsync(c->b.p, h_queries, (size_t)nq * 16, cudaMemcpyHostToDevice, st));
    RRTK_TRY(within_launch_f64(c->a.as<double>(), npts, c->b.as<double>(), nullptr, nq, r, cap, c->c.as<int32_t>(), c->d.as<int32_t>(), st));
    RRTK_CUDA(cudaMemcpyAsync(h_out, c->c.p, (size_t)nq * cap * 4, cudaMemcpyDeviceToHost, st));
    RRTK_CUDA(cudaMemcpyAsync(h_len, c->d.p, (size_t)nq * 4, cudaMemcpyDeviceToHost, st));
    RRTK_CUDA(cudaStreamSynchronize(st));
    return RRTK_OK;
}

// full ordering RRT.near returns (rrt.py:150-155), pinned stable
static int near_order_common(rrtk_ctx *c, int npts, int32_t *h_perm)
{
    cudaStream_t st = c->stream;
    RRTK_TRY(c->c.reserve((size_t)npts * 4));
    RRTK_TRY(c->d.reserve(argsort_scratch(npts)));
    RRTK_TRY(argsort_launch(c->b.as<int64_t>(), npts, c->c.as<int32_t>(), c->d.p, c->d.cap, st));
    RRTK_CUDA(cudaMemcpyAsync(h_perm, c->c.p, (size_t)npts * 4, cudaMemcpyDeviceToHost, st));
    RRTK_CUDA(cudaStreamSynchronize(st));
    return RRTK_OK;
}
int rrtk_ctx_near_order(rrtk_ctx *c, const int32_t *h_pts, int npts, int qx, int qy, int32_t *h_perm)
{
    RRTK_REQUIRE(c && npts >= 1 && h_pts && h_perm, "rrtk_ctx_near_order: bad argument");
    RRTK_TRY(c->a.reserve((size_t)npts * 8));
    RRTK_TRY(c->b.reserve((size_t)npts * 8));
    RRTK_CUDA(cudaMemcpyAsync(c->a.p, h_pts, (size_t)npts * 8, cudaMemcpyHostToDevice, c->stream));
    RRTK_TRY(dist2_launch(c->a.as<int32_t>(), npts, qx, qy, c->b.as<int64_t>(), c->stream));
    return near_order_common(c, npts, h_perm);
}
int rrtk_ctx_near_order_f64(rrtk_ctx *c, const double *h_pts, int npts, double qx, double qy, int32_t *h_perm)
{
    RRTK_REQUIRE(c && npts >= 1 && h_pts && h_perm, "rrtk_ctx_near_order_f64: bad argument");
    RRTK_TRY(c->a.reserve((size_t)npts * 16));
    RRTK_TRY(c->b.reserve((size_t)npts * 8));
    RRTK_CUDA(cudaMemcpyAsync(c->a.p, h_pts, (size_t)npts * 16, cudaMemcpyHostToDevice, c->stream));
    // non-negative doubles order like their bit patterns, so the int64 sorter applies
    RRTK_TRY(dist_launch_f64(c->a.as<double>(), npts, qx, qy, c->b.as<double>(), c->stream));
    return near_order_common(c, npts, h_perm);
}

// ---- K8: rewire / Dubins planners and the Dubins primitive ----------------------------------------------
static int check_plan2_cfg(const rrtk_plan2_cfg *cfg)
{
    RRTK_REQUIRE(cfg, "rrtk_plan2: null configuration");
    RRTK_REQUIRE(cfg->model == RRTK_MODEL_EUCLID || cfg->model == RRTK_MODEL_DUBINS, "rrtk_plan2: unknown model");
    RRTK_REQUIRE(cfg->r_rewire == cfg->r_rewire, "rrtk_plan2: NaN radius");
    RRTK_REQUIRE(!cfg->informed || cfg->r_goal == cfg->r_goal, "rrtk_plan2: NaN goal radius");
    RRTK_REQUIRE(!cfg->dubins_table || (cfg->table_radius >= 1 && cfg->table_radius <= 1024), "rrtk_plan2: table_radius out of range");
    if (cfg->model == RRTK_MODEL_DUBINS) {
        RRTK_REQUIRE(cfg->nheadings >= 1 && cfg->nheadings <= 255, "rrtk_plan2: need 1 <= nheadings <= 255");
        RRTK_REQUIRE(cfg->rho > 0.0 && cfg->rho <= 16384.0 && cfg->ds >= 0.05 && cfg->ds <= 16384.0,
                     "rrtk_plan2: need 0 < rho <= 16384 and 0.05 <= ds <= 16384 (cells)");
    }
    return RRTK_OK;
}

static int check_dubins_args(int nheadings, double rho, double ds)
{
    RRTK_REQUIRE(nheadings >= 1 && nheadings <= 255, "dubins: need 1 <= nheadings <= 255");
    // bounds keep the number of sampled points per path finite and sane (a path is at most ~ W + H + 19 rho long)
    RRTK_REQUIRE(rho > 0.0 && rho <= 16384.0 && ds >= 0.05 && ds <= 16384.0, "dubins: need 0 < rho <= 16384 and 0.05 <= ds <= 16384 (cells)");
    return RRTK_OK;
}

size_t rrtk_dubins_table_bytes(int radius, int nheadings)
{
    return (radius < 1 || radius > 1024 || nheadings < 1 || nheadings > 255) ? 0 : dubins_table_bytes(radius, nheadings);
}

int rrtk_dubins_table_build(int radius, int nheadings, double rho, void *d_table, void *stream)
{
    RRTK_REQUIRE(d_table && radius >= 1 && radius <= 1024, "rrtk_dubins_table_build: need a table and 1 <= radius <= 1024");
    RRTK_TRY(check_dubins_args(nheadings, rho, 1.0));
    DevInfo *d;
    RRTK_TRY(dev_info(&d));
    return dubins_table_launch(radius, nheadings, rho, d_table, d->sms, (cudaStream_t)stream);
}

size_t rrtk_plan2_scratch_bytes(int nplans, int n) { return (nplans < 0 || n < 1) ? 0 : plan2_scratch_bytes(nplans, n); }

int rrtk_plan2_batch(const rrtk_plan2_cfg *cfg, const uint32_t *d_bits, int W, int H, const rrtk_plan_desc *d_plans, int nplans, int n,
                     const int16_t *d_samples, const uint8_t *d_heads, int16_t *d_pts, uint8_t *d_head, double *d_cost, double *d_elen,
                     int32_t *d_parent, int64_t *d_stats, void *d_scratch, int threads, void *stream)
{
    RRTK_TRY(check_plan2_cfg(cfg));
    RRTK_REQUIRE(d_bits && d_plans && d_samples && d_pts && d_head && d_cost && d_elen && d_parent && d_stats && d_scratch,
                 "rrtk_plan2_batch: null pointer");
    RRTK_REQUIRE(nplans >= 0 && n >= 1 && n <= 65534, "rrtk_plan2_batch: need nplans >= 0 and 1 <= n <= 65534");
    RRTK_TRY(check_grid_dims(W, H, 16384));
    if (nplans == 0) return RRTK_OK;
    DevInfo *d;
    RRTK_TRY(dev_info(&d));
    return plan2_launch(*cfg, d_bits, W, H, d_plans, nplans, n, d_samples, d_heads, d_pts, d_head, d_cost, d_elen, d_parent, d_stats,
                        d_scratch, threads, d->optin, (cudaStream_t)stream);
}

int rrtk_plan2_footprint(int n, int threads, int *smem_bytes, int *blocks_per_sm)
{
    RRTK_REQUIRE(n >= 1 && n <= 65534, "rrtk_plan2_footprint: need 1 <= n <= 65534");
    DevInfo *d;
    RRTK_TRY(dev_info(&d));
    int rc = plan2_footprint(n, threads, d->optin, d->sm_smem, smem_bytes, blocks_per_sm);
    if (rc) set_error("plan with n=%d does not fit shared memory", n);
    return rc;
}

int rrtk_dubins_paths(const int32_t *d_q, int64_t nq, int nheadings, double rho, int32_t *d_word, double *d_tpq, double *d_len,
                      void *stream)
{
    RRTK_REQUIRE(d_q && nq >= 0, "rrtk_dubins_paths: bad argument");
    RRTK_TRY(check_dubins_args(nheadings, rho, 1.0));
    if (nq == 0) return RRTK_OK;
    return dubins_paths_launch(d_q, nq, nheadings, rho, d_word, d_tpq, d_len, (cudaStream_t)stream);
}

int rrtk_dubins_collision(const uint32_t *d_bits, int W, int H, const int32_t *d_q, const int32_t *d_world, int64_t nq, int nheadings,
                          double rho, double ds, uint8_t *d_free, void *stream)
{
    RRTK_REQUIRE(d_bits && d_q && d_free && nq >= 0, "rrtk_dubins_collision: bad argument");
    RRTK_TRY(check_dubins_args(nheadings, rho, ds));
    RRTK_TRY(check_grid_dims(W, H, 16384));
    if (nq == 0) return RRTK_OK;
    return dubins_walk_launch(d_bits, W, H, d_q, d_world, nq, nheadings, rho, ds, d_free, 0, nullptr, nullptr, (cudaStream_t)stream);
}

int rrtk_dubins_sample(const int32_t *d_q, int64_t nq, int nheadings, double rho, double ds, int cap, double *d_xyth, int32_t *d_count,
                       void *stream)
{
    RRTK_REQUIRE(d_q && d_xyth && d_count && nq >= 0 && cap >= 1, "rrtk_dubins_sample: bad argument");
    RRTK_TRY(check_dubins_args(nheadings, rho, ds));
    if (nq == 0) return RRTK_OK;
    return dubins_walk_launch(nullptr, 1, 1, d_q, nullptr, nq, nheadings, rho, ds, nullptr, cap, d_xyth, d_count, (cudaStream_t)stream);
}

// memo of the Dubins primitive over the rewire radius, kept in the context while (radius, headings, rho) stay the same
static int ctx_dubins_memo(rrtk_ctx *c, rrtk_plan2_cfg *use, cudaStream_t st)
{
    if (!(use->model == RRTK_MODEL_DUBINS && use->star && !use->dubins_table && use->r_rewire >= 1.0 && use->r_rewire <= 1024.0)) return RRTK_OK;
    const int R = (int)ceil(use->r_rewire);
    const size_t bytes = dubins_table_bytes(R, use->nheadings);
    if (bytes > ((size_t)256 << 20)) return RRTK_OK;
    if (c->dt_R != R || c->dt_NH != use->nheadings || c->dt_rho != use->rho || !c->dtable.p) {
        RRTK_CUDA(cudaStreamSynchronize(st));
        RRTK_TRY(c->dtable.reserve(bytes));
        RRTK_TRY(rrtk_dubins_table_build(R, use->nheadings, use->rho, c->dtable.p, st));
        RRTK_CUDA(cudaStreamSynchronize(st));
        c->dt_R = R; c->dt_NH = use->nheadings; c->dt_rho = use->rho;
    }
    use->dubins_table = c->dtable.p;
    use->table_radius = R;
    return RRTK_OK;
}

int rrtk_ctx_plan2(rrtk_ctx *c, const rrtk_plan2_cfg *cfg, const rrtk_plan_desc *h_plans, int nplans, int n, const int16_t *h_samples,
                   const uint64_t *h_state, const uint8_t *h_heads, int16_t *h_pts, uint8_t *h_head, double *h_cost, double *h_elen,
                   int32_t *h_parent, int64_t *h_stats)
{
    RRTK_TRY(check_plan2_cfg(cfg));
    RRTK_REQUIRE(c && h_plans && h_pts && h_head && h_cost && h_elen && h_parent && h_stats, "rrtk_ctx_plan2: null pointer");
    RRTK_REQUIRE(c->nworlds > 0, "rrtk_ctx_plan2: call rrtk_ctx_set_grids first");
    RRTK_REQUIRE((h_samples != nullptr) != (h_state != nullptr), "rrtk_ctx_plan2: pass exactly one of h_samples / h_state");
    RRTK_REQUIRE(nplans >= 0 && n >= 1 && n <= 65534, "rrtk_ctx_plan2: need nplans >= 0 and 1 <= n <= 65534");
    if (nplans == 0) return RRTK_OK;
    const bool dub = cfg->model == RRTK_MODEL_DUBINS;
    for (int p = 0; p < nplans; ++p) {
        const rrtk_plan_desc &d = h_plans[p];
        if (d.world < 0 || d.world >= c->nworlds || d.start_x < 0 || d.start_x >= c->W || d.goal_x < 0 || d.goal_x >= c->W ||
            d.start_y < 0 || d.start_y >= c->H || d.goal_y < 0 || d.goal_y >= c->H) {
            set_error("plan %d: world index or start/goal outside the grid", p);
            return RRTK_ERR_INVALID;
        }
        if (dub && (d.reserved[0] < 0 || d.reserved[0] >= cfg->nheadings || d.reserved[1] < 0 || d.reserved[1] >= cfg->nheadings)) {
            set_error("plan %d: start / goal heading outside [0, %d)", p, cfg->nheadings);
            return RRTK_ERR_INVALID;
        }
    }
    if (h_state) RRTK_TRY(require_free_cells(c, h_plans, nplans, "rrtk_ctx_plan2"));
    const size_t total = (size_t)nplans * n;
    if (h_samples)
        for (size_t i = 0; i < total; ++i) {
            const int x = h_samples[2 * i], y = h_samples[2 * i + 1];
            if (x < 0 || x >= c->W || y < 0 || y >= c->H) {
                set_error("sample %zu of plan %zu lies outside the grid", i % n, i / n);
                return RRTK_ERR_INVALID;
            }
        }
    if (dub && h_heads)
        for (size_t i = 0; i < total; ++i)
            if (h_heads[i] >= cfg->nheadings) {
                set_error("heading of sample %zu of plan %zu outside [0, %d)", i % n, i / n, cfg->nheadings);
                return RRTK_ERR_INVALID;
            }
    const size_t rows = (size_t)nplans * (n + 1);
    cudaStream_t st = c->stream;
    RRTK_TRY(c->plans.reserve(sizeof(rrtk_plan_desc) * nplans));
    RRTK_TRY(c->samples.reserve(total * 4));
    RRTK_TRY(c->heads.reserve(total));
    RRTK_TRY(c->pts.reserve(rows * 4));
    RRTK_TRY(c->head_out.reserve(rows));
    RRTK_TRY(c->cost.reserve(rows * 8));
    RRTK_TRY(c->elen.reserve(rows * 8));
    RRTK_TRY(c->parent.reserve(rows * 4));
    RRTK_TRY(c->stats.reserve((size_t)nplans * RRTK_STAT_COUNT * 8));
    RRTK_TRY(c->scratch2.reserve(plan2_scratch_bytes(nplans, n)));
    RRTK_CUDA(cudaMemcpyAsync(c->plans.p, h_plans, sizeof(rrtk_plan_desc) * nplans, cudaMemcpyHostToDevice, st));
    if (h_samples) {
        RRTK_CUDA(cudaMemcpyAsync(c->samples.p, h_samples, total * 4, cudaMemcpyHostToDevice, st));
    } else {
        DevInfo *d;
        RRTK_TRY(dev_info(&d));
        RRTK_TRY(c->state.reserve((size_t)nplans * 32));
        RRTK_CUDA(cudaMemcpyAsync(c->state.p, h_state, (size_t)nplans * 32, cudaMemcpyHostToDevice, st));
        RRTK_TRY(sample_streams_launch(c->bits.as<uint32_t>(), c->rowcum.as<int32_t>(), c->W, c->H, c->plans.as<rrtk_plan_desc>(),
                                       nplans, c->state.as<uint64_t>(), n, c->samples.as<int16_t>(), d->optin, st));
    }
    if (h_heads) RRTK_CUDA(cudaMemcpyAsync(c->heads.p, h_heads, total, cudaMemcpyHostToDevice, st));
    rrtk_plan2_cfg use = *cfg;
    RRTK_TRY(ctx_dubins_memo(c, &use, st));
    // informed: the unit-disc draws and the ellipse budgets are host arrays in this form of the call
    const double *h_balls = cfg->informed ? cfg->balls : nullptr;
    double *h_ell = cfg->informed ? cfg->ell_c : nullptr;
    use.balls = nullptr; use.ell_c = nullptr;
    if (h_balls) {
        RRTK_TRY(c->balls.reserve(total * 16));
        RRTK_CUDA(cudaMemcpyAsync(c->balls.p, h_balls, total * 16, cudaMemcpyHostToDevice, st));
        use.balls = c->balls.as<double>();
    }
    if (h_ell) {
        RRTK_TRY(c->ell.reserve(rows * 8));
        use.ell_c = c->ell.as<double>();
    }
    cfg = &use;
    RRTK_TRY(rrtk_plan2_batch(cfg, c->bits.as<uint32_t>(), c->W, c->H, c->plans.as<rrtk_plan_desc>(), nplans, n, c->samples.as<int16_t>(),
                              h_heads ? c->heads.as<uint8_t>() : nullptr, c->pts.as<int16_t>(), c->head_out.as<uint8_t>(),
                              c->cost.as<double>(), c->elen.as<double>(), c->parent.as<int32_t>(), c->stats.as<int64_t>(),
                              c->scratch2.p, 0, st));
    RRTK_CUDA(cudaMemcpyAsync(h_pts, c->pts.p, rows * 4, cudaMemcpyDeviceToHost, st));
    RRTK_CUDA(cudaMemcpyAsync(h_head, c->head_out.p, rows, cudaMemcpyDeviceToHost, st));
    RRTK_CUDA(cudaMemcpyAsync(h_cost, c->cost.p, rows * 8, cudaMemcpyDeviceToHost, st));
    RRTK_CUDA(cudaMemcpyAsync(h_elen, c->elen.p, rows * 8, cudaMemcpyDeviceToHost, st));
    RRTK_CUDA(cudaMemcpyAsync(h_parent, c->parent.p, rows * 4, cudaMemcpyDeviceToHost, st));
    RRTK_CUDA(cudaMemcpyAsync(h_stats, c->stats.p, (size_t)nplans * RRTK_STAT_COUNT * 8, cudaMemcpyDeviceToHost, st));
    if (h_ell) RRTK_CUDA(cudaMemcpyAsync(h_ell, c->ell.p, rows * 8, cudaMemcpyDeviceToHost, st));
    RRTK_CUDA(cudaStreamSynchronize(st));
    for (int p = 0; p < nplans; ++p)
        if (h_stats[(size_t)p * RRTK_STAT_COUNT + RRTK_STAT2_OVERFLOW]) {
            set_error("plan %d: a rewire-radius set exceeded the kernel's list (1024 vertices); reduce r_rewire", p);
            return RRTK_ERR_CAPACITY;
        }
    return RRTK_OK;
}

// K8 from host buffers with the worlds in the same call, chunked and pipelined like rrtk_ctx_plan_worlds2
int rrtk_ctx_plan2_worlds(rrtk_ctx *c, const rrtk_plan2_cfg *cfg, const void *h_grids, int nworlds, int W, int H, const rrtk_plan_desc *h_plans,
                          int nplans, int n, const int16_t *h_samples, const uint64_t *h_state, const uint8_t *h_heads, int flags, int path_cap,
                          int16_t *h_pts, uint8_t *h_head, double *h_cost, double *h_elen, int32_t *h_parent, int64_t *h_stats, int32_t *h_path,
                          int16_t *h_xy, uint8_t *h_path_head, int32_t *h_len, double *h_path_cost, int chunk_plans)
{
    const bool in_bits = flags & RRTK_IN_BITS, out_trees = flags & RRTK_OUT_TREES, out_paths = flags & RRTK_OUT_PATHS;
    const bool seed_balls = flags & RRTK_SEED_BALLS;
    RRTK_TRY(check_plan2_cfg(cfg));
    RRTK_REQUIRE(!seed_balls || h_state, "rrtk_ctx_plan2_worlds: RRTK_SEED_BALLS needs seed mode (h_state)");
    RRTK_REQUIRE(!seed_balls || cfg->informed, "rrtk_ctx_plan2_worlds: RRTK_SEED_BALLS needs cfg->informed");
    RRTK_REQUIRE(!seed_balls || !cfg->balls, "rrtk_ctx_plan2_worlds: RRTK_SEED_BALLS draws the unit-disc stream itself (pass cfg->balls = NULL)");
    RRTK_REQUIRE(c && h_grids && h_plans && h_stats, "rrtk_ctx_plan2_worlds: null pointer");
    RRTK_REQUIRE(!out_trees || (h_pts && h_head && h_cost && h_elen && h_parent),
                 "rrtk_ctx_plan2_worlds: RRTK_OUT_TREES needs h_pts, h_head, h_cost, h_elen, h_parent");
    RRTK_REQUIRE(!out_paths || (h_path && h_xy && h_len && h_path_cost && path_cap >= 1),
                 "rrtk_ctx_plan2_worlds: RRTK_OUT_PATHS needs h_path, h_xy, h_len, h_path_cost and path_cap >= 1");
    RRTK_REQUIRE((h_samples != nullptr) != (h_state != nullptr), "rrtk_ctx_plan2_worlds: pass exactly one of h_samples / h_state");
    RRTK_REQUIRE(nworlds >= 1 && nplans >= 0 && n >= 1 && n <= 65534, "rrtk_ctx_plan2_worlds: need nworlds >= 1, nplans >= 0, 1 <= n <= 65534");
    RRTK_TRY(check_grid_dims(W, H, 16384));
    if (nplans == 0) return RRTK_OK;
    const bool dub = cfg->model == RRTK_MODEL_DUBINS;
    for (int p = 0; p < nplans; ++p) {
        const rrtk_plan_desc &d = h_plans[p];
        if (d.world < 0 || d.world >= nworlds || d.start_x < 0 || d.start_x >= W || d.goal_x < 0 || d.goal_x >= W ||
            d.start_y < 0 || d.start_y >= H || d.goal_y < 0 || d.goal_y >= H) {
            set_error("plan %d: world index or start/goal outside the grid", p);
            return RRTK_ERR_INVALID;
        }
        if (p && d.world < h_plans[p - 1].world) {
            set_error("rrtk_ctx_plan2_worlds: plans must be ordered by world index (plan %d)", p);
            return RRTK_ERR_INVALID;
        }
        if (dub && (d.reserved[0] < 0 || d.reserved[0] >= cfg->nheadings || d.reserved[1] < 0 || d.reserved[1] >= cfg->nheadings)) {
            set_error("plan %d: start / goal heading outside [0, %d)", p, cfg->nheadings);
            return RRTK_ERR_INVALID;
        }
    }
    const size_t total = (size_t)nplans * n;
    if (h_samples)
        for (size_t i = 0; i < total; ++i) {
            const int x = h_samples[2 * i], y = h_samples[2 * i + 1];
            if (x < 0 || x >= W || y < 0 || y >= H) {
                set_error("sample %zu of plan %zu lies outside the grid", i % n, i / n);
                return RRTK_ERR_INVALID;
            }
        }
    if (dub && h_heads)
        for (size_t i = 0; i < total; ++i)
            if (h_heads[i] >= cfg->nheadings) {
                set_error("heading of sample %zu of plan %zu outside [0, %d)", i % n, i / n, cfg->nheadings);
                return RRTK_ERR_INVALID;
            }
    DevInfo *di;
    RRTK_TRY(dev_info(&di));
    if (chunk_plans <= 0) {
        // a plan of this kernel runs for tens of milliseconds: one block per SM and chunk keeps every copy hidden behind the
        // plans of the chunks before it, and the first chunk is on the device after 1/16 of the uploads
        chunk_plans = di->sms;
    }
    rrtk_plan2_cfg use = *cfg;
    RRTK_TRY(ctx_dubins_memo(c, &use, c->stream));
    const double *h_balls = cfg->informed ? cfg->balls : nullptr;      // host arrays in this form of the call
    double *h_ell = cfg->informed ? cfg->ell_c : nullptr;
    use.balls = nullptr; use.ell_c = nullptr;
    const size_t cells = (size_t)W * H, words = grid_words(W, H), rows1 = (size_t)n + 1;
    const size_t grid_bytes = in_bits ? words * 4 : cells;
    std::vector<int> starts;
    for (int p0 = 0; p0 < nplans; p0 += chunk_plans) starts.push_back(p0);
    starts.push_back(nplans);
    size_t max_m = 0, max_nw = 0;
    for (size_t k = 0; k + 1 < starts.size(); ++k) {
        const size_t m = (size_t)(starts[k + 1] - starts[k]);
        const size_t nw = (size_t)(h_plans[starts[k + 1] - 1].world - h_plans[starts[k]].world + 1);
        max_m = m > max_m ? m : max_m;
        max_nw = nw > max_nw ? nw : max_nw;
    }
    int status = RRTK_OK;
    auto cuda_ok = [&](cudaError_t e, const char *what) {
        if (e != cudaSuccess && status == RRTK_OK) status = cuda_fail(e, what);
        return e == cudaSuccess;
    };
    auto rrtk_ok = [&](int rc) {
        if (rc != RRTK_OK && status == RRTK_OK) status = rc;
        return rc == RRTK_OK;
    };
    if (h_state) RRTK_TRY(pipe_nfree_reserve(c, (size_t)nworlds));
    const size_t nslots = starts.size() - 1 < (size_t)kPipeSlots ? starts.size() - 1 : (size_t)kPipeSlots;
    for (size_t k = 0; k < nslots && status == RRTK_OK; ++k) {
        PipeSlot &s = c->pipe[k];
        if (!rrtk_ok(pipe_slot_init(c, s))) break;
        bool ok = rrtk_ok(s.bits.reserve(words * 4 * max_nw)) && rrtk_ok(s.rowcum.reserve((size_t)(W + 1) * 4 * max_nw)) &&
                  rrtk_ok(s.plans.reserve(sizeof(rrtk_plan_desc) * max_m)) && rrtk_ok(s.samples.reserve(max_m * n * 4)) &&
                  rrtk_ok(s.state.reserve(max_m * 32)) && rrtk_ok(s.heads.reserve(max_m * n)) && rrtk_ok(s.pts.reserve(rows1 * max_m * 4)) &&
                  rrtk_ok(s.head_out.reserve(rows1 * max_m)) && rrtk_ok(s.cost.reserve(rows1 * max_m * 8)) &&
                  rrtk_ok(s.elen.reserve(rows1 * max_m * 8)) && rrtk_ok(s.parent.reserve(rows1 * max_m * 4)) &&
                  rrtk_ok(s.stats.reserve(max_m * RRTK_STAT_COUNT * 8)) && rrtk_ok(s.scratch2.reserve(plan2_scratch_bytes((int)max_m, n)));
        if (ok && !in_bits) ok = rrtk_ok(s.og.reserve(cells * max_nw));
        if (ok && (h_balls || seed_balls)) ok = rrtk_ok(s.balls.reserve(max_m * n * 16));
        if (ok && h_ell) ok = rrtk_ok(s.ell.reserve(rows1 * max_m * 8));
        if (ok && out_paths)
            ok = rrtk_ok(s.path.reserve(max_m * path_cap * 4)) && rrtk_ok(s.xy.reserve(max_m * path_cap * 4)) &&
                 rrtk_ok(s.phead.reserve(max_m * path_cap)) && rrtk_ok(s.len.reserve(max_m * 4)) && rrtk_ok(s.pcost.reserve(max_m * 8));
    }
    for (size_t ci = 0; ci + 1 < starts.size() && status == RRTK_OK; ++ci) {
        const int p0 = starts[ci], m = starts[ci + 1] - starts[ci];
        PipeSlot &s = c->pipe[ci % kPipeSlots];
        cudaStream_t st = c->pipe_prep;
        if (ci >= (size_t)kPipeSlots && !cuda_ok(cudaStreamWaitEvent(st, s.done, 0), "cudaStreamWaitEvent")) break;
        const int w0 = h_plans[p0].world, w1 = h_plans[p0 + m - 1].world, nw = w1 - w0 + 1;
        const uint8_t *src = static_cast<const uint8_t *>(h_grids) + grid_bytes * w0;
        if (in_bits) {
            if (!cuda_ok(cudaMemcpyAsync(s.bits.p, src, grid_bytes * nw, cudaMemcpyHostToDevice, st), "cudaMemcpyAsync(bits)")) break;
        } else {
            if (!cuda_ok(cudaMemcpyAsync(s.og.p, src, grid_bytes * nw, cudaMemcpyHostToDevice, st), "cudaMemcpyAsync(og)")) break;
            if (!rrtk_ok(pack_launch(s.og.as<uint8_t>(), nw, W, H, s.bits.as<uint32_t>(), st))) break;
        }
        s.desc.assign(h_plans + p0, h_plans + p0 + m);
        for (rrtk_plan_desc &d : s.desc) d.world -= w0;
        if (!cuda_ok(cudaMemcpyAsync(s.plans.p, s.desc.data(), sizeof(rrtk_plan_desc) * m, cudaMemcpyHostToDevice, st), "cudaMemcpyAsync(plans)")) break;
        if (h_samples) {
            if (!cuda_ok(cudaMemcpyAsync(s.samples.p, h_samples + (size_t)p0 * n * 2, (size_t)m * n * 4, cudaMemcpyHostToDevice, st), "cudaMemcpyAsync(samples)")) break;
        } else {
            if (!rrtk_ok(free_rows_launch(s.bits.as<uint32_t>(), nw, W, H, s.rowcum.as<int32_t>(), st))) break;
            if (!cuda_ok(cudaMemcpy2DAsync(c->pin_nfree + w0, 4, s.rowcum.as<int32_t>() + W, (size_t)(W + 1) * 4, 4, nw, cudaMemcpyDeviceToHost, st),
                           "cudaMemcpy2DAsync(nfree)")) break;
            if (!cuda_ok(cudaMemcpyAsync(s.state.p, h_state + (size_t)p0 * 4, (size_t)m * 32, cudaMemcpyHostToDevice, st), "cudaMemcpyAsync(state)")) break;
            if (!rrtk_ok(sample_streams_launch(s.bits.as<uint32_t>(), s.rowcum.as<int32_t>(), W, H, s.plans.as<rrtk_plan_desc>(), m,
                                               s.state.as<uint64_t>(), n, s.samples.as<int16_t>(), di->optin, st))) break;
        }
        if (h_heads && !cuda_ok(cudaMemcpyAsync(s.heads.p, h_heads + (size_t)p0 * n, (size_t)m * n, cudaMemcpyHostToDevice, st), "cudaMemcpyAsync(heads)")) break;
        if (h_balls && !cuda_ok(cudaMemcpyAsync(s.balls.p, h_balls + (size_t)p0 * n * 2, (size_t)m * n * 16, cudaMemcpyHostToDevice, st), "cudaMemcpyAsync(balls)")) break;
        if (!cuda_ok(cudaEventRecord(s.ready, st), "cudaEventRecord")) break;
        st = s.stream;
        if (!cuda_ok(cudaStreamWaitEvent(st, s.ready, 0), "cudaStreamWaitEvent")) break;
        use.ell_c = h_ell ? s.ell.as<double>() : nullptr;
        if (seed_balls) {
            // probe (stops at the first solution vertex), then the unit-disc stream from the generator past that iteration
            use.balls = nullptr;
            if (!rrtk_ok(rrtk_plan2_batch(&use, s.bits.as<uint32_t>(), W, H, s.plans.as<rrtk_plan_desc>(), m, n, s.samples.as<int16_t>(),
                                          h_heads ? s.heads.as<uint8_t>() : nullptr, s.pts.as<int16_t>(), s.head_out.as<uint8_t>(), s.cost.as<double>(),
                                          s.elen.as<double>(), s.parent.as<int32_t>(), s.stats.as<int64_t>(), s.scratch2.p, 0, st))) break;
            if (!rrtk_ok(ball_streams_launch(s.rowcum.as<int32_t>(), W, s.plans.as<rrtk_plan_desc>(), m, n, s.state.as<uint64_t>(), nullptr,
                                             s.stats.as<int64_t>() + RRTK_STAT2_FIRST_SOL, RRTK_STAT_COUNT, s.balls.as<double>(), nullptr,
                                             nullptr, st))) break;
        }
        use.balls = (h_balls || seed_balls) ? s.balls.as<double>() : nullptr;
        if (!rrtk_ok(rrtk_plan2_batch(&use, s.bits.as<uint32_t>(), W, H, s.plans.as<rrtk_plan_desc>(), m, n, s.samples.as<int16_t>(),
                                      h_heads ? s.heads.as<uint8_t>() : nullptr, s.pts.as<int16_t>(), s.head_out.as<uint8_t>(), s.cost.as<double>(),
                                      s.elen.as<double>(), s.parent.as<int32_t>(), s.stats.as<int64_t>(), s.scratch2.p, 0, st))) break;
        if (!cuda_ok(cudaEventRecord(s.planned, st), "cudaEventRecord")) break;
        st = c->pipe_post;
        if (!cuda_ok(cudaStreamWaitEvent(st, s.planned, 0), "cudaStreamWaitEvent")) break;
        bool ok = true;
        if (out_paths) {
            ok = rrtk_ok(paths_xy_launch(s.parent.as<int32_t>(), s.pts.as<int16_t>(), s.cost.as<double>(), s.stats.as<int64_t>(), m, n, path_cap,
                                         s.path.as<int32_t>(), s.xy.as<int16_t>(), s.len.as<int32_t>(), s.pcost.as<double>(), st)) &&
                 cuda_ok(cudaMemcpyAsync(h_path + (size_t)p0 * path_cap, s.path.p, (size_t)m * path_cap * 4, cudaMemcpyDeviceToHost, st), "cudaMemcpyAsync(path)") &&
                 cuda_ok(cudaMemcpyAsync(h_xy + (size_t)p0 * path_cap * 2, s.xy.p, (size_t)m * path_cap * 4, cudaMemcpyDeviceToHost, st), "cudaMemcpyAsync(xy)") &&
                 cuda_ok(cudaMemcpyAsync(h_len + p0, s.len.p, (size_t)m * 4, cudaMemcpyDeviceToHost, st), "cudaMemcpyAsync(len)") &&
                 cuda_ok(cudaMemcpyAsync(h_path_cost + p0, s.pcost.p, (size_t)m * 8, cudaMemcpyDeviceToHost, st), "cudaMemcpyAsync(path_cost)");
            if (ok && h_path_head)
                ok = rrtk_ok(path_heads_launch(s.path.as<int32_t>(), s.head_out.as<uint8_t>(), m, n, path_cap, s.phead.as<uint8_t>(), st)) &&
                     cuda_ok(cudaMemcpyAsync(h_path_head + (size_t)p0 * path_cap, s.phead.p, (size_t)m * path_cap, cudaMemcpyDeviceToHost, st), "cudaMemcpyAsync(path_head)");
        }
        if (ok && out_trees)
            ok = cuda_ok(cudaMemcpyAsync(h_pts + (size_t)p0 * rows1 * 2, s.pts.p, rows1 * m * 4, cudaMemcpyDeviceToHost, st), "cudaMemcpyAsync(pts)") &&
                 cuda_ok(cudaMemcpyAsync(h_head + (size_t)p0 * rows1, s.head_out.p, rows1 * m, cudaMemcpyDeviceToHost, st), "cudaMemcpyAsync(head)") &&
                 cuda_ok(cudaMemcpyAsync(h_cost + (size_t)p0 * rows1, s.cost.p, rows1 * m * 8, cudaMemcpyDeviceToHost, st), "cudaMemcpyAsync(cost)") &&
                 cuda_ok(cudaMemcpyAsync(h_elen + (size_t)p0 * rows1, s.elen.p, rows1 * m * 8, cudaMemcpyDeviceToHost, st), "cudaMemcpyAsync(elen)") &&
                 cuda_ok(cudaMemcpyAsync(h_parent + (size_t)p0 * rows1, s.parent.p, rows1 * m * 4, cudaMemcpyDeviceToHost, st), "cudaMemcpyAsync(parent)");
        if (ok && h_ell) ok = cuda_ok(cudaMemcpyAsync(h_ell + (size_t)p0 * rows1, s.ell.p, rows1 * m * 8, cudaMemcpyDeviceToHost, st), "cudaMemcpyAsync(ell)");
        if (ok) cuda_ok(cudaMemcpyAsync(h_stats + (size_t)p0 * RRTK_STAT_COUNT, s.stats.p, (size_t)m * RRTK_STAT_COUNT * 8, cudaMemcpyDeviceToHost, st), "cudaMemcpyAsync(stats)");
        cuda_ok(cudaEventRecord(s.done, st), "cudaEventRecord");
    }
    pipe_drain(c, &status);
    if (status != RRTK_OK) return status;
    if (h_state) RRTK_TRY(pipe_require_free_cells(c, h_plans, nplans, "rrtk_ctx_plan2_worlds"));
    if (seed_balls) RRTK_TRY(pipe_require_rotations(h_plans, h_stats, nplans, RRTK_STAT2_FIRST_SOL, "rrtk_ctx_plan2_worlds"));
    for (int p = 0; p < nplans; ++p)
        if (h_stats[(size_t)p * RRTK_STAT_COUNT + RRTK_STAT2_OVERFLOW]) {
            set_error("plan %d: a rewire-radius set exceeded the kernel's list (1024 vertices); reduce r_rewire", p);
            return RRTK_ERR_CAPACITY;
        }
    return RRTK_OK;
}

int rrtk_ctx_dubins_paths(rrtk_ctx *c, const int32_t *h_q, int64_t nq, int nheadings, double rho, int32_t *h_word, double *h_tpq,
                          double *h_len)
{
    RRTK_REQUIRE(c && h_q && nq >= 0, "rrtk_ctx_dubins_paths: bad argument");
    if (nq == 0) return RRTK_OK;
    RRTK_TRY(c->a.reserve((size_t)nq * 24));
    RRTK_TRY(c->b.reserve((size_t)nq * 4));
    RRTK_TRY(c->c.reserve((size_t)nq * 24));
    RRTK_TRY(c->d.reserve((size_t)nq * 8));
    RRTK_CUDA(cudaMemcpyAsync(c->a.p, h_q, (size_t)nq * 24, cudaMemcpyHostToDevice, c->stream));
    RRTK_TRY(rrtk_dubins_paths(c->a.as<int32_t>(), nq, nheadings, rho, c->b.as<int32_t>(), c->c.as<double>(), c->d.as<double>(), c->stream));
    if (h_word) RRTK_CUDA(cudaMemcpyAsync(h_word, c->b.p, (size_t)nq * 4, cudaMemcpyDeviceToHost, c->stream));
    if (h_tpq) RRTK_CUDA(cudaMemcpyAsync(h_tpq, c->c.p, (size_t)nq * 24, cudaMemcpyDeviceToHost, c->stream));
    if (h_len) RRTK_CUDA(cudaMemcpyAsync(h_len, c->d.p, (size_t)nq * 8, cudaMemcpyDeviceToHost, c->stream));
    RRTK_CUDA(cudaStreamSynchronize(c->stream));
    return RRTK_OK;
}

static int check_dubins_queries(const rrtk_ctx *c, const int32_t *h_q, int64_t nq, int nheadings, bool in_grid)
{
    for (int64_t i = 0; i < nq; ++i) {
        const int32_t *e = h_q + 6 * i;
        if (e[2] < 0 || e[2] >= nheadings || e[5] < 0 || e[5] >= nheadings) {
            set_error("dubins query %lld: heading outside [0, %d)", (long long)i, nheadings);
            return RRTK_ERR_INVALID;
        }
        if (in_grid && (e[0] < 0 || e[0] >= c->W || e[3] < 0 || e[3] >= c->W || e[1] < 0 || e[1] >= c->H || e[4] < 0 || e[4] >= c->H)) {
            set_error("dubins query %lld: end point outside the grid", (long long)i);
            return RRTK_ERR_INVALID;
        }
    }
    return RRTK_OK;
}

int rrtk_ctx_dubins_collision(rrtk_ctx *c, int world, const int32_t *h_q, int64_t nq, int nheadings, double rho, double ds,
                              uint8_t *h_free)
{
    RRTK_REQUIRE(c && h_q && h_free && nq >= 0, "rrtk_ctx_dubins_collision: bad argument");
    RRTK_REQUIRE(c->nworlds > 0 && world >= 0 && world < c->nworlds, "rrtk_ctx_dubins_collision: no such world (rrtk_ctx_set_grids first)");
    RRTK_TRY(check_dubins_args(nheadings, rho, ds));
    RRTK_TRY(check_dubins_queries(c, h_q, nq, nheadings, true));
    if (nq == 0) return RRTK_OK;
    RRTK_TRY(c->a.reserve((size_t)nq * 24));
    RRTK_TRY(c->b.reserve((size_t)nq));
    RRTK_CUDA(cudaMemcpyAsync(c->a.p, h_q, (size_t)nq * 24, cudaMemcpyHostToDevice, c->stream));
    RRTK_TRY(rrtk_dubins_collision(c->bits.as<uint32_t>() + (size_t)world * grid_words(c->W, c->H), c->W, c->H, c->a.as<int32_t>(), nullptr,
                                   nq, nheadings, rho, ds, c->b.as<uint8_t>(), c->stream));
    RRTK_CUDA(cudaMemcpyAsync(h_free, c->b.p, (size_t)nq, cudaMemcpyDeviceToHost, c->stream));
    RRTK_CUDA(cudaStreamSynchronize(c->stream));
    return RRTK_OK;
}

int rrtk_ctx_dubins_sample(rrtk_ctx *c, const int32_t *h_q, int64_t nq, int nheadings, double rho, double ds, int cap, double *h_xyth,
                           int32_t *h_count)
{
    RRTK_REQUIRE(c && h_q && h_xyth && h_count && nq >= 0 && cap >= 1, "rrtk_ctx_dubins_sample: bad argument");
    RRTK_TRY(check_dubins_args(nheadings, rho, ds));
    RRTK_TRY(check_dubins_queries(c, h_q, nq, nheadings, false));
    if (nq == 0) return RRTK_OK;
    RRTK_TRY(c->a.reserve((size_t)nq * 24));
    RRTK_TRY(c->b.reserve((size_t)nq * cap * 24));
    RRTK_TRY(c->c.reserve((size_t)nq * 4));
    RRTK_CUDA(cudaMemcpyAsync(c->a.p, h_q, (size_t)nq * 24, cudaMemcpyHostToDevice, c->stream));
    RRTK_CUDA(cudaMemsetAsync(c->b.p, 0, (size_t)nq * cap * 24, c->stream));
    RRTK_TRY(rrtk_dubins_sample(c->a.as<int32_t>(), nq, nheadings, rho, ds, cap, c->b.as<double>(), c->c.as<int32_t>(), c->stream));
    RRTK_CUDA(cudaMemcpyAsync(h_xyth, c->b.p, (size_t)nq * cap * 24, cudaMemcpyDeviceToHost, c->stream));
    RRTK_CUDA(cudaMemcpyAsync(h_count, c->c.p, (size_t)nq * 4, cudaMemcpyDeviceToHost, c->stream));
    RRTK_CUDA(cudaStreamSynchronize(c->stream));
    return RRTK_OK;
}

}  // extern "C"
