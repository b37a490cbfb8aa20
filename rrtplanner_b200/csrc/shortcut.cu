// Greedy line-of-sight shortcut of path records (include/rrtk.h rrtk_shortcut_paths), one warp per path.
//
// For the kept point q_i the warp tries the later points q_{m-1}, q_{m-2}, ... in turn and keeps the first one the walk
// q_i -> q_k of RRT.collisionfree (rrt.py:183-229) finds free, or q_{i+1} when none is: farthest first, so the first free
// candidate is the greatest free index.  Every verdict is warp_first_hit on the grid through L1/L2 -- the walk the plan
// kernels run -- and always from the earlier point to the later one, the direction the tree's edges were walked.
// The row's points are staged in shared memory (packed x | y << 16) because every candidate is read once per kept point;
// the grid is not: one cfg3 world is 32 KB and one path reads a small part of it.
//
// The row is rewritten in place by lane 0.  Kept entry t comes from input index keep[t] >= t, and every later read is at an
// index above keep[t], so no read sees an entry already rewritten: points come from the staged copy, path ids from the row.
#include "common.cuh"

namespace rrtk {

constexpr int kScWarps = 4;              // paths per block

__global__ void __launch_bounds__(kScWarps * 32) shortcut_kernel(const uint32_t *__restrict__ bits, size_t words_per, int TY,
                                                                 const int *__restrict__ world, int world_stride, int npaths, int cap,
                                                                 short2 *xy, int *len, int *path, int *keep, double *cost)
{
    extern __shared__ uint32_t s_pts[];                                  // kScWarps x cap packed points
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int p = blockIdx.x * kScWarps + warp;
    if (p >= npaths) return;                                             // warp-uniform
    const int m = len[p];
    if (m <= 0 || m > cap) return;                                       // row left unwritten by rrtk_extract_paths_xy: untouched
    uint32_t *s = s_pts + (size_t)warp * cap;
    short2 *row = xy + (size_t)p * cap;
    int *prow = path ? path + (size_t)p * cap : nullptr;
    int *krow = keep ? keep + (size_t)p * cap : nullptr;
    for (int k = lane; k < m; k += 32) {
        const short2 v = row[k];
        s[k] = pack_xy(v.x, v.y);
    }
    __syncwarp();
    const GlobalGrid g{bits + (world ? (size_t)__ldg(world + (size_t)p * world_stride) * words_per : 0)};
    uint32_t a = s[0];
    int i = 0, t = 1;
    double c = 0.0;
    if (lane == 0 && krow) krow[0] = 0;
    while (i < m - 1) {
        int k = m - 1;
        for (; k > i + 1; --k) {
            const uint32_t b = s[k];
            if (warp_first_hit(g, TY, px(a), py(a), px(b), py(b), lane) < 0) break;
        }
        const uint32_t b = s[k];
        if (lane == 0) {
            row[t] = make_short2((short)px(b), (short)py(b));
            if (prow) prow[t] = prow[k];
            if (krow) krow[t] = k;
            c = reach_cost(c, dist2(b, px(a), py(a)));                   // the tree's cost sum: sqrt then add, left to right
        }
        ++t;
        i = k;
        a = b;
    }
    for (int q = t + lane; q < cap; q += 32) {
        row[q] = make_short2(-32768, -32768);
        if (prow) prow[q] = -1;
        if (krow) krow[q] = -1;
    }
    if (lane == 0) {
        len[p] = t;
        if (cost) cost[p] = c;
    }
}

// world: per-path world index at world[p * world_stride] (NULL = world 0); the pipelined plan call passes the world field
// of its rrtk_plan_desc array (stride 16 ints)
int shortcut_launch(const uint32_t *d_bits, int W, int H, const int32_t *d_world, int world_stride, int npaths, int cap, int16_t *d_xy,
                    int32_t *d_len, int32_t *d_path, int32_t *d_keep, double *d_cost, cudaStream_t st)
{
    if (npaths == 0) return RRTK_OK;
    const size_t smem = (size_t)kScWarps * cap * 4;
    if (smem > 48 * 1024) RRTK_CUDA(cudaFuncSetAttribute(shortcut_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    shortcut_kernel<<<(unsigned)((npaths + kScWarps - 1) / kScWarps), kScWarps * 32, smem, st>>>(
        d_bits, grid_words(W, H), tiles_y(H), d_world, world_stride, npaths, cap, reinterpret_cast<short2 *>(d_xy), d_len, d_path, d_keep,
        d_cost);
    RRTK_CUDA(cudaGetLastError());
    return RRTK_OK;
}

}  // namespace rrtk
