// Configuration space of a body with a heading (include/rrtk.h, rrtk_inflate_body): layer l of world w blocks cell c iff some
// offset d of stencil l has c + d inside the grid and og[c + d] != 0, i.e.
//     layer[l] = scipy.ndimage.binary_dilation(og != 0, structure = S_l[::-1, ::-1], border_value = 0)
// and the projection blocks a cell iff every layer blocks it.  A stencil arrives as runs (dx, dy_lo, dy_hi): the maximal runs of
// set cells of its rows.  Along y a run is an OR over hi - lo + 1 consecutive source bits, which two log-doubling levels
//     A_p[y] = any(src[y .. y + 2^p - 1]),   p = floor(log2(hi - lo + 1))
// answer exactly: run(x, y) = A_p(x + dx, y + lo) | A_p(x + dx, y + hi - 2^p + 1).
//
// One block per (world, 32-row x tile, kTyBlock words of y): it stages the source rows x0 - k .. x0 + 31 + k and the words
// ty0 - hw .. ty0 + kTyBlock - 1 + hw (hw = ceil(k / 32)) of its world once, builds the levels it needs in shared memory (row
// index fastest, so the 32 lanes of a warp -- 32 consecutive rows x -- never share a bank), and then writes every layer from
// them: per run four shared-memory reads, two funnel shifts and two ORs per output word.  The projection is an AND in registers.
#include "common.cuh"

namespace rrtk {

namespace {

constexpr int kTyBlock = 8;            // output words along y per block: one warp each

__device__ __forceinline__ uint32_t inside_bits(int ty, int H)
{
    const int valid = H - ty * 32;
    return valid >= 32 ? 0xffffffffu : (valid <= 0 ? 0u : ((1u << valid) - 1u));
}

}  // namespace

// levels [P][NW + 1][R]: R staged rows, NW staged words (+ one zero word so that a funnel shift never reads past the end)
__global__ void __launch_bounds__(32 * kTyBlock) inflate_body_kernel(const uint32_t *__restrict__ bits, int W, int H, int k, int P,
                                                                    const int32_t *__restrict__ runs,
                                                                    const int32_t *__restrict__ layer_runs, int nlayers,
                                                                    uint32_t *__restrict__ layers, uint32_t *__restrict__ proj)
{
    extern __shared__ uint32_t lev[];
    const int TX = tiles_x(W), TY = tiles_y(H);
    const int nty = (TY + kTyBlock - 1) / kTyBlock;
    const int world = blockIdx.x / (TX * nty);
    const int rem = blockIdx.x - world * TX * nty;
    const int tx = rem / nty, ty0 = (rem - (rem / nty) * nty) * kTyBlock;
    const int hw = (k + 31) >> 5;
    const int R = 32 + 2 * k, NW = kTyBlock + 2 * hw, NW1 = NW + 1;
    const int x0 = tx * 32;
    const size_t wpg = grid_words(W, H);
    const uint32_t *src = bits + (size_t)world * wpg;

    // ---- stage level 0: the source words, cells outside the grid free --------------------------------------
    for (int i = threadIdx.x; i < NW1 * R; i += blockDim.x) {
        const int wj = i / R, r = i - wj * R;
        const int x = x0 - k + r, ty = ty0 - hw + wj;
        uint32_t v = 0u;
        if (wj < NW && x >= 0 && x < W && ty >= 0 && ty < TY) v = __ldg(src + word_index(x, ty * 32, TY)) & inside_bits(ty, H);
        lev[i] = v;
    }
    __syncthreads();
    // ---- level p from level p - 1: A_p[y] = A_{p-1}[y] | A_{p-1}[y + 2^(p-1)] --------------------------------
    for (int p = 1; p < P; ++p) {
        const uint32_t *a = lev + (size_t)(p - 1) * NW1 * R;
        uint32_t *b = lev + (size_t)p * NW1 * R;
        const int s = 1 << (p - 1), sw = s >> 5, sb = s & 31;
        for (int i = threadIdx.x; i < NW1 * R; i += blockDim.x) {
            const int wj = i / R, r = i - wj * R;
            const int j0 = wj + sw, j1 = j0 + 1;
            const uint32_t lo = j0 < NW1 ? a[j0 * R + r] : 0u, hi = j1 < NW1 ? a[j1 * R + r] : 0u;
            b[i] = a[i] | __funnelshift_r(lo, hi, sb);
        }
        __syncthreads();
    }

    // ---- every layer from the staged levels ------------------------------------------------------------------
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int x = x0 + lane, ty = ty0 + warp;
    if (ty >= TY) return;
    const uint32_t pad = x < W ? ~inside_bits(ty, H) : 0xffffffffu;     // padding cells stay set, as the packer leaves them
    const int ybase = (warp + hw) * 32;                                  // staged bit position of the output word's first cell
    const uint32_t oi = word_index(x, ty * 32, TY);
    uint32_t all = 0xffffffffu;
    for (int l = 0; l < nlayers; ++l) {
        const int r0 = __ldg(layer_runs + l), r1 = __ldg(layer_runs + l + 1);
        uint32_t acc = 0u;
        for (int r = r0; r < r1; ++r) {
            const int dx = __ldg(runs + 3 * r), lo = __ldg(runs + 3 * r + 1), hi = __ldg(runs + 3 * r + 2);
            const int p = 31 - __clz(hi - lo + 1);
            const uint32_t *b = lev + (size_t)p * NW1 * R + (lane + k + dx);
            const int q1 = ybase + lo, q2 = ybase + hi - (1 << p) + 1;
            const uint32_t a1 = __funnelshift_r(b[(q1 >> 5) * R], b[((q1 >> 5) + 1) * R], q1 & 31);
            const uint32_t a2 = __funnelshift_r(b[(q2 >> 5) * R], b[((q2 >> 5) + 1) * R], q2 & 31);
            acc |= a1 | a2;
        }
        acc |= pad;
        layers[((size_t)world * nlayers + l) * wpg + oi] = acc;
        all &= acc;
    }
    if (proj) proj[(size_t)world * wpg + oi] = all;
}

// Staged extent of a run set: k = largest |dx|, |dy_lo|, |dy_hi|, P = levels needed (floor(log2(longest run)) + 1).
size_t body_smem_bytes(int k, int P)
{
    const int hw = (k + 31) >> 5;
    return sizeof(uint32_t) * (size_t)P * (kTyBlock + 2 * hw + 1) * (32 + 2 * k);
}

int body_launch(const uint32_t *d_bits, int nworlds, int W, int H, const int32_t *d_runs, const int32_t *d_layer_runs, int nlayers, int k,
                int P, uint32_t *d_layers, uint32_t *d_proj, cudaStream_t st)
{
    if (nworlds == 0) return RRTK_OK;
    const size_t smem = body_smem_bytes(k, P);
    RRTK_CUDA(cudaFuncSetAttribute(inflate_body_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const size_t blocks = (size_t)nworlds * tiles_x(W) * ((tiles_y(H) + kTyBlock - 1) / kTyBlock);
    if (blocks > 0x7fffffffu) {
        set_error("rrtk_inflate_body: %zu thread blocks exceed one launch", blocks);
        return RRTK_ERR_CAPACITY;
    }
    inflate_body_kernel<<<(unsigned)blocks, 32 * kTyBlock, smem, st>>>(d_bits, W, H, k, P, d_runs, d_layer_runs, nlayers, d_layers, d_proj);
    RRTK_CUDA(cudaGetLastError());
    return RRTK_OK;
}

}  // namespace rrtk
