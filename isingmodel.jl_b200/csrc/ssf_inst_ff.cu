#include "ssf_inst.cuh"
namespace isb {
cudaError_t launch_ssf_ff(const SsfParams &p, int npl, bool list, bool tma, int grid, int threads, size_t smem,
                          cudaStream_t st) {
    return launch_pair<float, float>(p, npl, list, tma, grid, threads, smem, st);
}
}  // namespace isb
