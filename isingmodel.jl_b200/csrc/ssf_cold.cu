// ssf_cold.cu — the sweep kernel for the COLD part of an anneal (few accepted flips): local fields in shared memory.
//
// ssf_kernel keeps a chain's N Float64 fields in registers (64 per thread at N = 1024): 14 chains per SM, two waves for
// the 4096 replicas of BASELINE config 2, 3.5 warps per scheduler — and a 32-site window is a chain of ~170 DEPENDENT
// instructions (noise word, schedule, the Float64 decision), so the cold sweeps are latency-bound.  Once flips are rare the
// fields hardly change: here they live in shared memory (8 KiB per chain, in the permuted order of a J row, so that
// applying a row is a lane-private 128-bit read-modify-write), a thread needs ~50 registers, 28 chains fit one SM (ONE wave
// for config 2) and seven warps per scheduler hide each other's latencies.  Same arithmetic, same decisions:
//   * the window logic (32-site speculation, first flip applied, later lanes re-evaluated) is ssf_kernel's sequential path
//     (src/SingleSpinFlip.jl:31-36,46-55,65-74 one site at a time; src/SamplingHelper.jl:45-49 the step loop);
//   * the incremental field update `fields += +-2 J[i, :]` uses the same operations on the same values, so the cached
//     fields stay bit-identical to ssf_kernel's and the launches of a segmented run can alternate freely;
//   * one Philox4x32-10 block per lane serves 128 consecutive steps (the same words as philox_step_word_k).
// ssf_run_device selects this kernel per segment (csrc/ssf.cu) when the previous segment's acceptance is low and the run
// needs nothing the kernel leaves out: sequential order, no traces, no near-tie guard or audit; Float64 fields and
// couplings, or (FIXED) the int32 fixed-point ones of the same run.
#include <stdint.h>

#include "common.cuh"
#include "handles.hpp"
#include "ssf_kernel.cuh"

namespace isb {

constexpr int SSF_COLD_CHAINS = 28;

// FIXED: the fixed-point variant (int32 fields and couplings, decisions as in ssf_kernel's int32 instantiation: integer
// thresholds, ssf_exact_field in between); the fields are packed by four, 4 KiB per chain at N = 1024.
template <bool FIXED>
__global__ void __launch_bounds__(32 * SSF_COLD_CHAINS, 1) ssf_cold_kernel(const SsfParams p) {
    using FT = typename std::conditional<FIXED, int32_t, double>::type;
    using FV = typename std::conditional<FIXED, int4, double2>::type;   // one 128-bit pack of fields / couplings
    constexpr int PK = FIXED ? 4 : 2;
    extern __shared__ __align__(16) unsigned char cold_smem[];
    constexpr uint32_t FULL = 0xffffffffu;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int r = blockIdx.x * p.nw + warp;
    if (warp >= p.nw || r >= p.R) return;
    const int npad = p.npad, npl = npad >> 5;       // npl is a multiple of PK (the host checks it)
    // F[(k / PK) * 32 PK + lane * PK + (k % PK)] = field of site k * 32 + lane (the permuted order of a J row)
    FT *F = reinterpret_cast<FT *>(cold_smem) + (size_t)warp * npad;
    const FT *Jg = reinterpret_cast<const FT *>(p.J);
    uint32_t sw = 0;
    {
        const FT *fr = reinterpret_cast<const FT *>(p.fields) + (int64_t)r * npad;
        const int8_t *sr = p.spins + (int64_t)r * p.lds;
        for (int k = 0; k < npl; ++k) {
            F[(k / PK) * (32 * PK) + lane * PK + (k % PK)] = fr[k * 32 + lane];
            sw |= (sr[k * 32 + lane] > 0 ? 1u : 0u) << k;
        }
    }
    const int rule = p.rule;
    const bool metro = rule == 2;
    const double tsc = p.tscale ? __ldg(&p.tscale[r]) : 1.0;
    unsigned long long nflips = 0, nfall = 0;
    const uint64_t spT = (uint64_t)p.steps_per_T;
    uint64_t ti = 0, tr = 0;                         // t = ti * spT + tr
    int64_t cached_ti = -1;
    double cachedT = 0.0;
    Philox4 blk{0, 0, 0, 0};                         // lane j: the words of steps 4 (cb + j) .. 4 (cb + j) + 3
    uint64_t cb = 0;
    bool have_blk = false;

    int64_t t = 0;
    int site = p.start;
    while (t < p.nsteps) {
        const int k = site >> 5, l_first = site & 31;
        int len = 32 - l_first;
        if (p.n - site < len) len = p.n - site;
        if (p.nsteps - t < len) len = (int)(p.nsteps - t);
        const int off = lane - l_first;
        const bool mine = off >= 0 && off < len;
        double Tl;                                   // temperature of my step (T <- schedule(k) before step k)
        {
            const uint64_t a_hi = tr + (uint64_t)(len - 1);
            if (a_hi < spT) {
                if ((int64_t)ti != cached_ti) {
                    cachedT = __dmul_rn(__ldg(&p.Tsched[ti]), tsc);
                    cached_ti = (int64_t)ti;
                }
                Tl = cachedT;
            } else {
                const uint64_t a = tr + (uint64_t)(mine ? off : 0);
                Tl = __dmul_rn(__ldg(&p.Tsched[ti + a / spT]), tsc);
            }
        }
        double f = 0.0;                              // fluctuation of my step
        if (rule != 0) {
            const int64_t tl = t + (mine ? off : 0);
            if (p.fluct_mode == 0) {
                const uint64_t g0 = p.step_offset + (uint64_t)t;
                if (!have_blk || ((g0 + 31) >> 2) >= cb + 32 || (g0 >> 2) < cb) {
                    cb = g0 >> 2;
                    const uint64_t q = cb + (uint64_t)lane;
                    blk = philox4x32_10k((uint32_t)q, (uint32_t)(q >> 32), (uint32_t)r, DOM_SSF_FLUCT << 28, p.keys);
                    have_blk = true;
                }
                const uint64_t gs = p.step_offset + (uint64_t)tl;
                const int src = (int)((gs >> 2) - cb);
                const uint32_t wx = __shfl_sync(FULL, blk.x, src), wy = __shfl_sync(FULL, blk.y, src);
                const uint32_t wz = __shfl_sync(FULL, blk.z, src), ww = __shfl_sync(FULL, blk.w, src);
                const uint32_t pick = (uint32_t)(gs & 3u);
                f = ssf_fluct_from_word(rule, pick == 0 ? wx : (pick == 1 ? wy : (pick == 2 ? wz : ww)));
            } else if (p.fluct_mode == 1) {
                f = __ldg(&p.fluct[tl]);
            } else {
                f = __ldg(&p.fluct[(int64_t)r * p.fluct_pitch + tl]);
            }
        }
        const double ftl = __dmul_rn(f, Tl);
        bool mybit = (sw >> k) & 1u;
        const int kpos = (k / PK) * (32 * PK) + lane * PK + (k % PK);
        FT hk = F[kpos];                             // my own site's field; mirrors F[kpos] through the window
        uint32_t rem = __ballot_sync(FULL, mine);
        auto fts = [&]() { return metro ? (mybit ? ftl : -ftl) : ftl; };
        [[maybe_unused]] int flo = 0, fhi = 0;
        if constexpr (FIXED)   // (my spin changes only when my turn in the window is over: fixed through the window)
            fixed_thresholds(fts(), p.hsign * __ldg(&p.hext[k * 32 + lane]), p.fix_q, p.fix_invq, p.fix_margin, flo, fhi);
        while (true) {
            bool nb;
            if constexpr (FIXED) {
                nb = hk >= fhi;
                const bool near = !nb && hk >= flo && ((rem >> lane) & 1u);
                const uint32_t nm = __ballot_sync(FULL, near);
                if (nm) {   // rare: decide on the reference's fresh sequential row dot
                    const double ex = ssf_exact_field(p.J64, p.ld64, p.hext, p.hsign, p.n, sw, k * 32 + lane, near);
                    if (near) nb = !(__dsub_rn(2.0 * ex, fts()) < 0.0);
                    nfall += __popc(nm);
                }
            } else {
                nb = !(__dsub_rn(2.0 * hk, fts()) < 0.0);   // heaviside(0) = 1, src/SpinSystems.jl:163-171
            }
            const uint32_t fm = __ballot_sync(FULL, nb != mybit) & rem;
            if (fm == 0) break;
            const int l0 = __ffs(fm) - 1;
            const uint32_t upto = (2u << l0) - 1u;   // lanes <= l0 (l0 == 31 -> all ones)
            const bool up = (__ballot_sync(FULL, nb) >> l0) & 1u;
            const FT d = up ? (FT)2 : (FT)-2;
            const FT *row = Jg + (int64_t)(k * 32 + l0) * p.ldj;
            hk += d * row[kpos];
            // fields += d * J[row]: every lane owns the positions c * 32 PK + lane * PK + {0 .. PK - 1} of its chain's
            // fields (four 128-bit row loads in flight per batch: the loop is a chain of L2 / L1 latencies otherwise)
            auto axpy = [&](FV &f, const FV &j) {
                if constexpr (FIXED) {
                    f.x += d * j.x;
                    f.y += d * j.y;
                    f.z += d * j.z;
                    f.w += d * j.w;
                } else {
                    f.x += d * j.x;
                    f.y += d * j.y;
                }
            };
            const int nc = npl / PK;
            int c = 0;
            for (; c + 4 <= nc; c += 4) {
                FV jv[4], fv[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) jv[u] = __ldg(reinterpret_cast<const FV *>(row + (c + u) * (32 * PK)) + lane);
#pragma unroll
                for (int u = 0; u < 4; ++u) fv[u] = *(reinterpret_cast<FV *>(F + (c + u) * (32 * PK)) + lane);
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    axpy(fv[u], jv[u]);
                    *(reinterpret_cast<FV *>(F + (c + u) * (32 * PK)) + lane) = fv[u];
                }
            }
            for (; c < nc; ++c) {
                const FV jv = __ldg(reinterpret_cast<const FV *>(row + c * (32 * PK)) + lane);
                FV *fp = reinterpret_cast<FV *>(F + c * (32 * PK)) + lane;
                FV fv = *fp;
                axpy(fv, jv);
                *fp = fv;
            }
            if (lane == l0) {
                sw ^= 1u << k;
                mybit = !mybit;
            }
            ++nflips;
            rem &= ~upto;
            if (rem == 0) break;
        }
        t += len;
        site += len;
        if (site >= p.n) site = 0;
        tr += (uint64_t)len;
        if (tr >= spT) {
            ti += tr / spT;
            tr %= spT;
        }
    }
    {
        FT *fr = reinterpret_cast<FT *>(p.fields) + (int64_t)r * npad;
        int8_t *sr = p.spins + (int64_t)r * p.lds;
        for (int k = 0; k < npl; ++k) {
            fr[k * 32 + lane] = F[(k / PK) * (32 * PK) + lane * PK + (k % PK)];
            if (k * 32 + lane < p.n) sr[k * 32 + lane] = ((sw >> k) & 1u) ? (int8_t)1 : (int8_t)-1;
        }
        if (lane == 0) {
            p.flips[r] = nflips;
            if (nfall) atomicAdd(p.fallbacks, nfall);
        }
    }
}

// chains per CTA the shared memory holds for this model (0: the kernel does not apply); fixed: the int32 variant
int ssf_cold_chains(const isb_ctx *ctx, int npad, bool fixed) {
    if (npad % (fixed ? 128 : 64) != 0) return 0;
    const size_t per_chain = (size_t)npad * (fixed ? sizeof(int32_t) : sizeof(double));
    return (int)std::min<size_t>(SSF_COLD_CHAINS, (ctx->smem_optin - 1024) / per_chain);
}

cudaError_t launch_ssf_cold(const SsfParams &p, int chains, bool fixed, cudaStream_t st) {
    SsfParams q = p;
    q.nw = chains;
    const size_t smem = (size_t)chains * p.npad * (fixed ? sizeof(int32_t) : sizeof(double));
    auto kern = fixed ? ssf_cold_kernel<true> : ssf_cold_kernel<false>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kern<<<(p.R + chains - 1) / chains, 32 * chains, smem, st>>>(q);
    return cudaGetLastError();
}

}  // namespace isb
