// ssf_inst.cuh — instantiates ssf_kernel for one (field type, coupling type) pair; included by
// ssf_inst_dd.cu (Float64 fields and couplings) / ssf_inst_ff.cu (float fields and couplings) / ssf_inst_ii.cu (int32
// fixed-point fields and couplings), compiled in parallel.
#pragma once
#include "ssf_kernel.cuh"

namespace isb {

template <typename K>
static cudaError_t launch_kernel(K kern, const SsfParams &p, int grid, int threads, size_t smem, cudaStream_t st) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kern<<<grid, threads, smem, st>>>(p);
    return cudaGetLastError();
}

template <typename HT, typename JT, int NPL>
static cudaError_t launch_one(const SsfParams &p, bool list, bool tma, int grid, int threads, size_t smem, cudaStream_t st) {
    auto go = [&](auto kern) { return launch_kernel(kern, p, grid, threads, smem, st); };
    if constexpr (std::is_same<HT, double>::value) {
        if (p.guard > 0.0) {   // couplings from a small non-dyadic alphabet: the instantiation with the near-tie guard
            if (list) return tma ? go(ssf_kernel<HT, JT, NPL, true, true, true>) : go(ssf_kernel<HT, JT, NPL, true, false, true>);
            return tma ? go(ssf_kernel<HT, JT, NPL, false, true, true>) : go(ssf_kernel<HT, JT, NPL, false, false, true>);
        }
    }
    if (list) return tma ? go(ssf_kernel<HT, JT, NPL, true, true>) : go(ssf_kernel<HT, JT, NPL, true, false>);
    return tma ? go(ssf_kernel<HT, JT, NPL, false, true>) : go(ssf_kernel<HT, JT, NPL, false, false>);
}

template <typename HT, typename JT>
static cudaError_t launch_pair(const SsfParams &p, int npl, bool list, bool tma, int grid, int threads, size_t smem,
                               cudaStream_t st) {
    switch (npl) {
        case 1: return launch_one<HT, JT, 1>(p, list, tma, grid, threads, smem, st);
        case 2: return launch_one<HT, JT, 2>(p, list, tma, grid, threads, smem, st);
        case 4: return launch_one<HT, JT, 4>(p, list, tma, grid, threads, smem, st);
        case 8: return launch_one<HT, JT, 8>(p, list, tma, grid, threads, smem, st);
        case 16: return launch_one<HT, JT, 16>(p, list, tma, grid, threads, smem, st);
        case 32: return launch_one<HT, JT, 32>(p, list, tma, grid, threads, smem, st);
        default: return cudaErrorInvalidValue;
    }
}

}  // namespace isb
