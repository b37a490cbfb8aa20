// One planner kind of the packed-key plan kernel per translation unit (compiled in parallel):
// the including .cu defines RRTK_SCAN_KIND and RRTK_SCAN_FN.
#include "plan_scan.cuh"

namespace rrtk {

template <int K, int T, int MB = ScanCfg<RRTK_SCAN_KIND, K, T>::kMinBlocks>
static int scan_launch_kt(const PlanParams &P, int nplans, size_t smem, cudaStream_t st)
{
    auto kern = plan_scan_kernel<RRTK_SCAN_KIND, K, T, MB>;
    RRTK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<nplans, T, smem, st>>>(P);
    RRTK_CUDA(cudaGetLastError());
    return RRTK_OK;
}

template <int K>
static int scan_launch_k(const PlanParams &P, int nplans, int T, int two_per_sm, size_t smem, cudaStream_t st)
{
    switch (T) {
        case 64: return scan_launch_kt<K, 64>(P, nplans, smem, st);
        case 128: return scan_launch_kt<K, 128>(P, nplans, smem, st);
        case 160: return scan_launch_kt<K, 160>(P, nplans, smem, st);
        case 256: return two_per_sm ? scan_launch_kt<K, 256, 2>(P, nplans, smem, st) : scan_launch_kt<K, 256>(P, nplans, smem, st);
        case 512: return scan_launch_kt<K, 512>(P, nplans, smem, st);
    }
    set_error("packed-key plan kernel: unsupported block size %d", T);
    return RRTK_ERR_INVALID;
}

// resident blocks per SM of the kernel that would run (registers, shared memory incl. the static part, threads): asked of the
// runtime, not estimated
template <int K, int T, int MB = ScanCfg<RRTK_SCAN_KIND, K, T>::kMinBlocks>
static int scan_occupancy_kt(size_t smem)
{
    auto kern = plan_scan_kernel<RRTK_SCAN_KIND, K, T, MB>;
    int blocks = 0;
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess ||
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks, kern, T, smem) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return blocks;
}

template <int K>
static int scan_occupancy_k(int T, int two_per_sm, size_t smem)
{
    switch (T) {
        case 64: return scan_occupancy_kt<K, 64>(smem);
        case 128: return scan_occupancy_kt<K, 128>(smem);
        case 160: return scan_occupancy_kt<K, 160>(smem);
        case 256: return two_per_sm ? scan_occupancy_kt<K, 256, 2>(smem) : scan_occupancy_kt<K, 256>(smem);
        case 512: return scan_occupancy_kt<K, 512>(smem);
    }
    return 0;
}

int RRTK_SCAN_OCC_FN(int T, int K, int two_per_sm, size_t smem)
{
    switch (K) {
        case 4: return scan_occupancy_k<4>(T, two_per_sm, smem);
        case 8: return scan_occupancy_k<8>(T, two_per_sm, smem);
        case 16: return scan_occupancy_k<16>(T, two_per_sm, smem);
    }
    return 0;
}

int RRTK_SCAN_FN(const PlanParams &P, int nplans, int T, int K, int two_per_sm, size_t smem, cudaStream_t st)
{
    switch (K) {
        case 4: return scan_launch_k<4>(P, nplans, T, two_per_sm, smem, st);
        case 8: return scan_launch_k<8>(P, nplans, T, two_per_sm, smem, st);
        case 16: return scan_launch_k<16>(P, nplans, T, two_per_sm, smem, st);
    }
    set_error("packed-key plan kernel: unsupported samples per round %d", K);
    return RRTK_ERR_INVALID;
}

}  // namespace rrtk
