#include "ssf_inst.cuh"
namespace isb {
cudaError_t launch_ssf_dd(const SsfParams &p, int npl, bool list, bool tma, int grid, int threads, size_t smem,
                          cudaStream_t st) {
    return launch_pair<double, double>(p, npl, list, tma, grid, threads, smem, st);
}
}  // namespace isb
