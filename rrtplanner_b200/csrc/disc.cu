// Configuration space of a disc-shaped robot (include/rrtk.h, rrtk_inflate_disc): cell (x, y) of the output is blocked iff
// some obstacle cell (u, v) inside the grid has (x - u)^2 + (y - v)^2 <= r2, distances between cell indices.  That is
// scipy.ndimage.binary_dilation(og != 0, structure = {(i, j): i^2 + j^2 <= r2}, border_value = 0), and with r2 =
// floor(rho * rho) the same as EDT^2 <= rho^2.
//
// An exact separable distance transform, so the time per cell does not depend on r2:
//   pass 1 (disc_rows_kernel, one warp per (world, row x)): g(x, y) = distance along y to the nearest obstacle of row x,
//          from __ffs / __clz on the tiled words and warp scans across them; stored as uint16 (65535 = none) in the
//          scratch, g[((world * W) + x) * TY * 32 + y].  Rows never hold more than 32768 cells, so 16 bits are exact.
//   pass 2 (disc_cols_kernel, one warp per (output, 32-cell y tile), lane = y): blocked(x, y) iff some row u has
//          (x - u)^2 + g(u, y)^2 <= r2, i.e. |x - u| <= h(u) = isqrt(r2 - g(u, y)^2).  Thresholding turns every parabola
//          of the lower envelope (Felzenszwalb-Huttenlocher) into an interval [u - h, u + h], and a cell is covered iff
//          max_{u <= x} (u + h(u)) >= x  or  min_{u >= x} (u - h(u)) <= x: one backward and one forward running extremum
//          per lane, no envelope stack.  A ballot per x forms the output word.
// The squared-distance field itself is never stored (it would take 4 bytes per cell).
#include <climits>

#include "common.cuh"

namespace rrtk {

namespace {

constexpr int kNoObstacle = 1 << 20;     // farther than any cell of a grid (sides <= 32768)

// bits of word ty that lie inside the grid's H cells
__device__ __forceinline__ uint32_t y_inside_bits(int ty, int H)
{
    const int valid = H - ty * 32;
    return valid >= 32 ? 0xffffffffu : (valid <= 0 ? 0u : ((1u << valid) - 1u));
}

// floor(sqrt(v)) for 0 <= v <= INT32_MAX: the fp32 estimate is within 0.01 of sqrt(v), one step corrects it
__device__ __forceinline__ int isqrt_i32(int v)
{
    int s = __float2int_rz(sqrtf(__int2float_rn(v)));
    const unsigned uv = (unsigned)v;
    if ((unsigned)s * (unsigned)s > uv) --s;
    else if ((unsigned)(s + 1) * (unsigned)(s + 1) <= uv) ++s;
    return s;
}

// half-width of the x interval that the nearest obstacle of row u, g cells away along y, blocks; -1: none
__device__ __forceinline__ int reach(int g, int r2, int rmax)
{
    return g > rmax ? -1 : isqrt_i32(r2 - g * g);
}

__global__ void __launch_bounds__(256) disc_rows_kernel(const uint32_t *__restrict__ bits, int nworlds, int W, int H,
                                                        uint16_t *__restrict__ g)
{
    const int lane = threadIdx.x & 31;
    const int TY = tiles_y(H), nchunks = (TY + 31) >> 5;      // TY <= 1024: at most 32 chunks of 32 words
    const size_t wpg = grid_words(W, H), rows = (size_t)nworlds * W;
    const size_t nwarps = ((size_t)gridDim.x * blockDim.x) >> 5;
    for (size_t row = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; row < rows; row += nwarps) {
        const int world = (int)(row / W), x = (int)(row - (size_t)world * W);
        const uint32_t *rw = bits + (size_t)world * wpg + (size_t)(x >> 5) * TY * 32 + (x & 31);   // word ty at rw[32 ty]
        uint16_t *gr = g + row * (size_t)TY * 32;
        // first obstacle of every chunk of 32 words; lane c keeps chunk c's
        int chunk_first = kNoObstacle;
        for (int c = 0; c < nchunks; ++c) {
            const int ty = c * 32 + lane;
            const uint32_t w = ty < TY ? __ldg(rw + (size_t)ty * 32) & y_inside_bits(ty, H) : 0u;
            int f = w ? ty * 32 + __ffs(w) - 1 : kNoObstacle;
            for (int o = 16; o; o >>= 1) f = min(f, __shfl_xor_sync(RRTK_FULL, f, o));
            if (lane == c) chunk_first = f;
        }
        int chunks_from = chunk_first;                        // first obstacle in chunks >= lane
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_down_sync(RRTK_FULL, chunks_from, o);
            if (lane + o < 32) chunks_from = min(chunks_from, v);
        }
        int carry = -kNoObstacle;                             // last obstacle in the chunks before c
        for (int c = 0; c < nchunks; ++c) {
            const int ty = c * 32 + lane;
            const uint32_t w = ty < TY ? __ldg(rw + (size_t)ty * 32) & y_inside_bits(ty, H) : 0u;
            int upto = w ? ty * 32 + 31 - __clz(w) : -kNoObstacle;      // inclusive prefix max over the chunk's words
            int from = w ? ty * 32 + __ffs(w) - 1 : kNoObstacle;        // inclusive suffix min
            for (int o = 1; o < 32; o <<= 1) {
                const int a = __shfl_up_sync(RRTK_FULL, upto, o), b = __shfl_down_sync(RRTK_FULL, from, o);
                if (lane >= o) upto = max(upto, a);
                if (lane + o < 32) from = min(from, b);
            }
            const int after = __shfl_sync(RRTK_FULL, chunks_from, (c + 1) & 31);
            int prev = __shfl_up_sync(RRTK_FULL, upto, 1), next = __shfl_down_sync(RRTK_FULL, from, 1);
            prev = max(lane == 0 ? -kNoObstacle : prev, carry);
            next = min(lane == 31 ? kNoObstacle : next, c + 1 < 32 ? after : kNoObstacle);
            carry = max(carry, __shfl_sync(RRTK_FULL, upto, 31));
            if (ty < TY) {
                uint32_t packed[16];
#pragma unroll
                for (int b = 0; b < 32; ++b) {
                    const int y = ty * 32 + b;
                    const uint32_t lo = w & (0xffffffffu >> (31 - b)), hi = w >> b;
                    const int p = lo ? ty * 32 + 31 - __clz(lo) : prev;
                    const int q = hi ? y + __ffs(hi) - 1 : next;
                    const uint32_t d = (uint32_t)min(min(y - p, q - y), 65535);
                    packed[b >> 1] = (b & 1) ? (packed[b >> 1] | (d << 16)) : d;
                }
                uint4 *dst = reinterpret_cast<uint4 *>(gr + (size_t)ty * 32);
#pragma unroll
                for (int k = 0; k < 4; ++k) dst[k] = make_uint4(packed[4 * k], packed[4 * k + 1], packed[4 * k + 2], packed[4 * k + 3]);
            }
        }
    }
}

__global__ void __launch_bounds__(256) disc_cols_kernel(const uint16_t *__restrict__ g, int nworlds, int W, int H,
                                                        const int32_t *__restrict__ src, const int32_t *__restrict__ r2s, int nout,
                                                        uint32_t *__restrict__ out)
{
    const int lane = threadIdx.x & 31;
    const int TX = tiles_x(W), TY = tiles_y(H);
    const size_t wpg = grid_words(W, H), jobs = (size_t)nout * TY, rstride = (size_t)TY * 32;
    const size_t nwarps = ((size_t)gridDim.x * blockDim.x) >> 5;
    for (size_t job = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; job < jobs; job += nwarps) {
        const int o = (int)(job / TY), ty = (int)(job - (size_t)o * TY);
        const int s = __ldg(src + o), r2 = __ldg(r2s + o);
        if (s < 0 || s >= nworlds || r2 < 0) continue;        // documented: such an output is left unwritten
        const uint16_t *gc = g + (size_t)s * W * rstride + (size_t)ty * 32 + lane;     // g(u, y) at gc[u * rstride]
        uint32_t *ow = out + (size_t)o * wpg + (size_t)ty * 32 + lane;                  // word of tile tx at ow[tx * rstride]
        const uint32_t pad = ~y_inside_bits(ty, H);
        const int rmax = isqrt_i32(r2);
        // backward: an obstacle row u >= x blocks x iff u - h(u) <= x
        int lo = INT_MAX;
        for (int tx = TX - 1; tx >= 0; --tx) {
            int gv[32];
#pragma unroll
            for (int xl = 0; xl < 32; ++xl) {
                const int u = tx * 32 + xl;
                gv[xl] = u < W ? (int)gc[(size_t)u * rstride] : 65535;
            }
            uint32_t mine = 0xffffffffu;                      // rows x >= W are padding: all set
#pragma unroll
            for (int xl = 31; xl >= 0; --xl) {
                const int u = tx * 32 + xl;
                if (u < W) {
                    lo = min(lo, u - reach(gv[xl], r2, rmax));
                    const uint32_t m = __ballot_sync(RRTK_FULL, lo <= u);
                    if (lane == xl) mine = m;
                }
            }
            ow[(size_t)tx * rstride] = mine;
        }
        // forward: an obstacle row u <= x blocks x iff u + h(u) >= x
        int hi = INT_MIN;
        for (int tx = 0; tx < TX; ++tx) {
            int gv[32];
#pragma unroll
            for (int xl = 0; xl < 32; ++xl) {
                const int u = tx * 32 + xl;
                gv[xl] = u < W ? (int)gc[(size_t)u * rstride] : 65535;
            }
            uint32_t mine = ow[(size_t)tx * rstride];
#pragma unroll
            for (int xl = 0; xl < 32; ++xl) {
                const int u = tx * 32 + xl;
                if (u < W) {
                    hi = max(hi, u + reach(gv[xl], r2, rmax));
                    const uint32_t m = __ballot_sync(RRTK_FULL, hi >= u);
                    if (lane == xl) mine |= m;
                }
            }
            ow[(size_t)tx * rstride] = mine | pad;
        }
    }
}

unsigned warp_blocks(size_t warps)
{
    size_t blocks = (warps + 7) / 8;                          // 8 warps per 256-thread block
    if (blocks > 148 * 32) blocks = 148 * 32;
    return (unsigned)(blocks ? blocks : 1);
}

}  // namespace

size_t disc_scratch_bytes(int nworlds, int W, int H) { return (size_t)nworlds * W * tiles_y(H) * 32 * sizeof(uint16_t); }

int disc_launch(const uint32_t *d_bits, int nworlds, int W, int H, const int32_t *d_src, const int32_t *d_r2, int nout,
                uint32_t *d_out, void *d_scratch, cudaStream_t st)
{
    if (nout == 0 || nworlds == 0) return RRTK_OK;
    uint16_t *g = static_cast<uint16_t *>(d_scratch);
    disc_rows_kernel<<<warp_blocks((size_t)nworlds * W), 256, 0, st>>>(d_bits, nworlds, W, H, g);
    disc_cols_kernel<<<warp_blocks((size_t)nout * tiles_y(H)), 256, 0, st>>>(g, nworlds, W, H, d_src, d_r2, nout, d_out);
    RRTK_CUDA(cudaGetLastError());
    return RRTK_OK;
}

}  // namespace rrtk
