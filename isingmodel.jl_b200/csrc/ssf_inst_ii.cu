#include "ssf_inst.cuh"
namespace isb {
// The fixed-point path (SsfParams::fix_q): sequential order, plain kernel (rows from L1 / L2; see ssf_run_device).
cudaError_t launch_ssf_ii(const SsfParams &p, int npl, int grid, int threads, cudaStream_t st) {
    auto go = [&](auto kern) { return launch_kernel(kern, p, grid, threads, 0, st); };
    switch (npl) {
        case 1: return go(ssf_kernel<int32_t, int32_t, 1, false, false>);
        case 2: return go(ssf_kernel<int32_t, int32_t, 2, false, false>);
        case 4: return go(ssf_kernel<int32_t, int32_t, 4, false, false>);
        case 8: return go(ssf_kernel<int32_t, int32_t, 8, false, false>);
        case 16: return go(ssf_kernel<int32_t, int32_t, 16, false, false>);
        case 32: return go(ssf_kernel<int32_t, int32_t, 32, false, false>);
        default: return cudaErrorInvalidValue;
    }
}
}  // namespace isb
