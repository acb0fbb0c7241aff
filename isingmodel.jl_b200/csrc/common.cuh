// common.cuh — device helpers shared by the sm_100a kernels of libising_b200.so:
// mbarrier / bulk-copy (TMA) PTX wrappers, warp reductions, Philox4x32-10 and the
// uniform -> fluctuation transforms that replace Distributions.jl's samplers
// (reference call sites: src/SamplingHelper.jl:24,40,105-106,121-122).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

namespace isb {

// ------------------------------------------------------------------ mbarrier + bulk async copy
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
    // make the initialised barriers visible to the async (TMA) proxy
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug traps (context error) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    uint32_t spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        if (++spins > (1u << 22)) __trap();
    }
}
// 1-D bulk copy global -> shared, completion signalled on an mbarrier (SASS: UBLKCP).
__device__ __forceinline__ void bulk_g2s(void *smem_dst, const void *gmem_src, uint32_t bytes, uint64_t *bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(smem_dst)),
        "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}

// ------------------------------------------------------------------ thread-block clusters
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// ------------------------------------------------------------------ warp helpers
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ int warp_sum_int(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ------------------------------------------------------------------ Philox4x32-10
// Salmon, Moraes, Dror, Shaw, SC'11.  Checked word for word against oracle/ and the Random123 known answers (tests/test_oracle.py, tests/test_gpu_parity.py::test_philox_raw_matches_oracle_and_kat).
struct Philox4 {
    uint32_t x, y, z, w;
};
__host__ __device__ __forceinline__ Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                          uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint64_t p0 = (uint64_t)0xD2511F53u * c0;
        const uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
        const uint32_t n1 = (uint32_t)p1;
        const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        const uint32_t n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    return Philox4{c0, c1, c2, c3};
}
// Same function with the ten round keys precomputed (they depend on the seed only): saves the 20 key-schedule
// additions per block in kernels that draw many blocks per thread.
struct PhiloxKeys {
    uint32_t k0[10], k1[10];
};
__host__ __device__ __forceinline__ PhiloxKeys philox_keys(uint64_t seed) {
    PhiloxKeys K;
    uint32_t a = (uint32_t)seed, b = (uint32_t)(seed >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        K.k0[r] = a;
        K.k1[r] = b;
        a += 0x9E3779B9u;
        b += 0xBB67AE85u;
    }
    return K;
}
__host__ __device__ __forceinline__ Philox4 philox4x32_10k(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                           const PhiloxKeys &K) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint64_t p0 = (uint64_t)0xD2511F53u * c0;
        const uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ K.k0[r];
        const uint32_t n1 = (uint32_t)p1;
        const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ K.k1[r];
        const uint32_t n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    }
    return Philox4{c0, c1, c2, c3};
}
__host__ __device__ __forceinline__ uint32_t philox_pick(const Philox4 &p, uint32_t w) {
    return w == 0 ? p.x : (w == 1 ? p.y : (w == 2 ? p.z : p.w));
}

// Stream domains (top 4 bits of counter word 3).
enum : uint32_t { DOM_SSF_FLUCT = 1, DOM_SSF_NODES = 2, DOM_BIP_VISIBLE = 3, DOM_BIP_HIDDEN = 4, DOM_PT_SWAP = 5,
                  DOM_PA_RESAMPLE = 6 };
// Replica-exchange decisions (isb_ssf_run_pt): word .x of counter (lo(K), hi(K), ladder, DOM_PT_SWAP<<28 | lo) decides the
// swap of levels (lo, lo+1) in that ladder after absolute round K.
// Population-annealing resampling (isb_ssf_run_pa): word .x of counter (lo(K), hi(K), population, DOM_PA_RESAMPLE<<28) is
// the offset U of the systematic resampling of that population after absolute temperature step K.

// Word assigned to step `step` of replica `replica` in a single-spin run:
// counter = (lo(step>>2), hi(step>>2), replica, domain<<28), key = seed, word = step & 3.
__host__ __device__ __forceinline__ uint32_t philox_step_word(uint64_t seed, uint32_t domain, uint32_t replica,
                                                              uint64_t step) {
    const uint64_t q = step >> 2;
    const Philox4 p = philox4x32_10((uint32_t)q, (uint32_t)(q >> 32), replica, domain << 28, (uint32_t)seed,
                                    (uint32_t)(seed >> 32));
    return philox_pick(p, (uint32_t)(step & 3));
}
__host__ __device__ __forceinline__ uint32_t philox_step_word_k(const PhiloxKeys &K, uint32_t domain, uint32_t replica,
                                                                uint64_t step) {
    const uint64_t q = step >> 2;
    const Philox4 p = philox4x32_10k((uint32_t)q, (uint32_t)(q >> 32), replica, domain << 28, K);
    return philox_pick(p, (uint32_t)(step & 3));
}
// Block of 4 words for units 4*uq .. 4*uq+3 of one layer at step `step` of replica `replica`
// (bipartite runs): counter = (lo(step), hi(step), replica, domain<<28 | uq).
__host__ __device__ __forceinline__ Philox4 philox_unit_block(uint64_t seed, uint32_t domain, uint32_t replica,
                                                              uint64_t step, uint32_t uq) {
    return philox4x32_10((uint32_t)step, (uint32_t)(step >> 32), replica, (domain << 28) | uq, (uint32_t)seed,
                         (uint32_t)(seed >> 32));
}

// u in (0,1): (w + 1/2) 2^-32, never 0 or 1; 1 - u = (~w + 1/2) 2^-32 exactly.
// The variates are evaluated in single precision with the hardware log2 (two MUFU) and returned as doubles:
// the Float64 decision arithmetic downstream is unchanged, the fluctuation itself carries ~2^-22 relative
// error, far below the 2^-32 granularity of u in the tails that matter.  isb_philox_*_fluct dump exactly these
// values, so parity tests feed the oracle the same doubles.
__device__ __forceinline__ float u_from_word_f(uint32_t w) {
    return fmaf((float)w, 2.3283064365386963e-10f, 1.1641532182693481e-10f);
}
// Logistic(0,1) by inversion: log(u / (1-u))   (GlauberDynamics / SCA: SingleSpinFlip.jl:43, OnBipartiteGraph.jl:15)
__device__ __forceinline__ double logistic_from_word(uint32_t w) {
    return (double)(0.69314718055994531f * (__log2f(u_from_word_f(w)) - __log2f(u_from_word_f(~w))));
}
// Exponential(1) by inversion: -log(u)         (MetropolisMethod / MomentumAnnealing: SingleSpinFlip.jl:62, OnBipartiteGraph.jl:50)
__device__ __forceinline__ double exponential_from_word(uint32_t w) {
    return (double)(-0.69314718055994531f * __log2f(u_from_word_f(w)));
}

// fluctuation of a rule from a word: rule ids follow ising_b200.h (0 Hopfield, 1 Glauber, 2 Metropolis)
__device__ __forceinline__ double ssf_fluct_from_word(int rule, uint32_t w) {
    return rule == 1 ? logistic_from_word(w) : (rule == 2 ? exponential_from_word(w) : 0.0);
}

// Uniform site in [0, n): high half of w * n (SamplingHelper.jl:23,39 draw rand(rng, 1:N)).
__host__ __device__ __forceinline__ int32_t node_from_word(uint32_t w, int n) {
    return (int32_t)(((uint64_t)w * (uint64_t)(uint32_t)n) >> 32);
}

}  // namespace isb
