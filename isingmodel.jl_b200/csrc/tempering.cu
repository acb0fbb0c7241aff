// tempering.cu — device-resident parallel tempering for single-spin ensembles (isb_ssf_run_pt): the round loop over the
// sweep dispatch of isb_ssf_run (ssf_sweep_device), the replica-exchange kernel and the replica-overlap kernel.  The sweep
// kernels are not touched: every round is exactly one traced isb_ssf_run of the same steps, and the exchange decides on the
// energies those kernels trace at the last step of the round.
#include <algorithm>

#include "common.cuh"
#include "handles.hpp"

namespace isb {

// One CTA per ladder g (replicas g*L .. g*L + L - 1).  level_of[r] = level held by replica r; levels[l] = temperature
// factor of level l.  Records the traced E / M of the round per level (the replica that held the level during the round),
// adds the round's flips into the run total, then decides the swaps of the round's parity, one pair per thread (the
// pairs (lo, lo + 1) of one parity are disjoint).
__global__ void pt_exchange_kernel(int L, int G, uint64_t K, uint64_t seed, const double *__restrict__ levels,
                                   int32_t *level_of, double *tscale, const double *__restrict__ Eround,
                                   const double *__restrict__ Mround, double *recE, double *recM,
                                   unsigned long long *accepted, const unsigned long long *__restrict__ flips,
                                   unsigned long long *flips_total) {
    extern __shared__ int slot_of[];   // [L]: slot of this ladder holding level l
    const int g = blockIdx.x;
    const int base = g * L;
    for (int s = threadIdx.x; s < L; s += blockDim.x) {
        slot_of[level_of[base + s]] = s;
        flips_total[base + s] += flips[base + s];
    }
    __syncthreads();
    for (int l = threadIdx.x; l < L; l += blockDim.x) {
        const int r = base + slot_of[l];
        if (recE) recE[(int64_t)l * G + g] = Eround[r];
        if (recM) recM[(int64_t)l * G + g] = Mround[r];
    }
    for (int lo = (int)(K & 1) + 2 * (int)threadIdx.x; lo + 1 < L; lo += 2 * (int)blockDim.x) {
        const int a = base + slot_of[lo], b = base + slot_of[lo + 1];
        // IEEE round-to-nearest operations, no contraction: a host replay of the rule reproduces d bit for bit
        const double d = __dmul_rn(__dsub_rn(__ddiv_rn(1.0, levels[lo]), __ddiv_rn(1.0, levels[lo + 1])),
                                   __dsub_rn(Eround[a], Eround[b]));
        const Philox4 w = philox4x32_10((uint32_t)K, (uint32_t)(K >> 32), (uint32_t)g, (DOM_PT_SWAP << 28) | (uint32_t)lo,
                                        (uint32_t)seed, (uint32_t)(seed >> 32));
        const double u = ((double)w.x + 0.5) * 2.3283064365386963e-10;   // (w + 1/2) 2^-32, exact
        if (d >= 0.0 || u < exp(d)) {
            level_of[a] = lo + 1;
            level_of[b] = lo;
            tscale[a] = levels[lo + 1];
            tscale[b] = levels[lo];
            atomicAdd(&accepted[lo], 1ull);
        }
    }
}

// Q[l][p] = (sum_i s_i^a s_i^b) / N between the replicas of ladders 2p and 2p+1 that held level l during the round
// (launched before the exchange).  Grid (L, G/2); the products are summed as integers (dp4a over 4 sites per word).
__global__ void pt_overlap_kernel(int L, int n, const int8_t *__restrict__ spins, int64_t lds,
                                  const int32_t *__restrict__ level_of, double *recQ) {
    __shared__ int ra, rb;
    __shared__ int part[32];
    const int l = blockIdx.x, p = blockIdx.y;
    const int ba = 2 * p * L, bb = (2 * p + 1) * L;
    for (int s = threadIdx.x; s < L; s += blockDim.x) {
        if (level_of[ba + s] == l) ra = ba + s;
        if (level_of[bb + s] == l) rb = bb + s;
    }
    __syncthreads();
    const int8_t *sa = spins + (int64_t)ra * lds, *sb = spins + (int64_t)rb * lds;   // rows are 32-byte aligned
    const int n4 = n >> 2;
    int acc = 0;
    for (int i = threadIdx.x; i < n4; i += blockDim.x)
        acc = __dp4a(reinterpret_cast<const int *>(sa)[i], reinterpret_cast<const int *>(sb)[i], acc);
    for (int i = 4 * n4 + threadIdx.x; i < n; i += blockDim.x) acc += (int)sa[i] * (int)sb[i];
    acc = warp_sum_int(acc);
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) part[w] = acc;
    __syncthreads();
    if (w == 0) {
        acc = lane < (int)(blockDim.x >> 5) ? part[lane] : 0;
        acc = warp_sum_int(acc);
        if (lane == 0) recQ[(int64_t)l * gridDim.y + p] = (double)acc / (double)n;
    }
}

int ssf_pt_run_device(isb_ens *e, int rule, int n_levels, const double *d_levels, int64_t rounds, int64_t steps_per_round,
                      int order, int start, uint64_t seed, uint64_t step_offset, uint64_t round_offset, int32_t *d_nodes,
                      const double *d_T, int32_t *d_level_of, double *d_Eround, double *d_Mround, double *d_recE,
                      double *d_recM, double *d_recQ, unsigned long long *d_accepted, unsigned long long *d_flips_total) {
    isb_model *m = e->model;
    isb_ctx *ctx = m->ctx;
    const int L = n_levels, G = e->R / n_levels;
    const int64_t n = m->n;
    const int xthreads = std::min(1024, (L + 31) / 32 * 32);
    for (int64_t k = 0; k < rounds; ++k) {
        const int64_t t0 = k * steps_per_round;
        const uint64_t so = step_offset + (uint64_t)t0;
        const int st = (int)(((int64_t)start + t0 % n) % n);
        if (int rc = ssf_sweep_device(e, rule, steps_per_round, order, d_nodes, st, ISB_FLUCT_PHILOX, nullptr, seed, so, d_T,
                                      steps_per_round, steps_per_round, d_Eround, d_Mround, nullptr))
            return rc;
        if (d_recQ) {
            pt_overlap_kernel<<<dim3(L, G / 2), 256, 0, ctx->stream>>>(L, m->n, e->spins, e->lds, d_level_of,
                                                                       d_recQ + k * (int64_t)L * (G / 2));
            ISB_CUDA(ctx, cudaGetLastError());
            e->last_launches += 1;
        }
        pt_exchange_kernel<<<G, xthreads, (size_t)L * sizeof(int), ctx->stream>>>(
            L, G, round_offset + (uint64_t)k, seed, d_levels, d_level_of, e->d_tscale, d_Eround, d_Mround,
            d_recE ? d_recE + k * (int64_t)e->R : nullptr, d_recM ? d_recM + k * (int64_t)e->R : nullptr, d_accepted,
            e->d_flips, d_flips_total);
        ISB_CUDA(ctx, cudaGetLastError());
        e->last_launches += 1;
    }
    return ISB_OK;
}

}  // namespace isb
