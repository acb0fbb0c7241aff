// population.cu — population annealing for single-spin ensembles (isb_ssf_run_pa) and the replica gather under it
// (isb_ens_select_replicas).  The sweep kernels are not touched: every temperature step is one traced isb_ssf_run of the
// same steps (ssf_sweep_device, the sweep dispatch of isb_ssf_run), and the resampling decides on the energies those
// kernels trace at the last step.  The resampling is a segmented multi-CTA scheme (PA_THREADS slots per CTA, up to
// PA_THREADS CTAs per population), so populations are not limited by shared memory:
//   pa_weight_kernel  a_r = -db E_r and the CTA maxima of a (and the per-slot flip totals)
//   pa_scan_kernel    population max, x_r = exp(a_r - max), W_r = floor(x_r 2^32), CTA-local inclusive scan of W, CTA
//                     sums of W and x
//   pa_parent_kernel  every child slot j finds its parent, the smallest r with C_r > t_j, by a binary search over the
//                     CTA sums and then the CTA-local scan (load-balanced however many copies one parent gets); family
//                     labels follow the parents; lnQ
//   gather_rows_kernel the state of slot parent(j) into slot j of the second buffers (ens_select_device)
#include <cub/block/block_reduce.cuh>
#include <cub/block/block_scan.cuh>

#include <algorithm>

#include "common.cuh"
#include "handles.hpp"

namespace isb {

constexpr int PA_THREADS = 1024;   // slots per CTA; a population of P <= 2^20 slots spans at most 1024 CTAs

struct MaxOp {
    __device__ __forceinline__ double operator()(double a, double b) const { return a > b ? a : b; }
};

// ------------------------------------------------------------------ replica gather
// dst row r of every buffer = src row from[r]; rows are a multiple of 16 bytes (N padded to 32 sites).
struct GatherRows {
    const uint4 *src[3];
    uint4 *dst[3];
    int words[3];   // 16-byte words per row
    int nbuf;
};

__global__ void gather_rows_kernel(GatherRows g, const int32_t *__restrict__ from, int R) {
    for (int r = blockIdx.x; r < R; r += gridDim.x) {
        const int64_t s = from[r];
#pragma unroll
        for (int b = 0; b < 3; ++b) {   // (a constant trip count keeps the parameter arrays out of local memory)
            if (b >= g.nbuf) break;
            const int w = g.words[b];
            const uint4 *__restrict__ in = g.src[b] + s * w;
            uint4 *__restrict__ out = g.dst[b] + (int64_t)r * w;
            for (int i = threadIdx.x; i < w; i += blockDim.x) out[i] = in[i];
        }
    }
}

int ens_select_device(isb_ens *e, const int32_t *d_src) {
    isb_model *m = e->model;
    isb_ctx *ctx = m->ctx;
    const size_t R = (size_t)e->R;
    const size_t fbytes = (size_t)m->npad * (m->fast_ok ? ssf_field_elem_size(m) : sizeof(double));
    const bool fields = e->fields_rule_sign != 0, ifields = e->ifields_ok;
    if (!e->spins2) ISB_CUDA(ctx, cudaMalloc(&e->spins2, R * e->lds));
    if (fields && !e->fields2) ISB_CUDA(ctx, cudaMalloc(&e->fields2, R * fbytes));
    if (ifields && !e->ifields2) ISB_CUDA(ctx, cudaMalloc(&e->ifields2, R * m->npad * sizeof(int32_t)));
    GatherRows g{};
    auto add = [&g](const void *src, void *dst, size_t bytes) {
        g.src[g.nbuf] = (const uint4 *)src;
        g.dst[g.nbuf] = (uint4 *)dst;
        g.words[g.nbuf] = (int)(bytes / 16);
        g.nbuf += 1;
    };
    add(e->spins, e->spins2, (size_t)e->lds);
    if (fields) add(e->fields, e->fields2, fbytes);
    if (ifields) add(e->ifields, e->ifields2, (size_t)m->npad * sizeof(int32_t));
    const int grid = (int)std::min<size_t>(R, (size_t)ctx->num_sms * 16);
    gather_rows_kernel<<<grid, 256, 0, ctx->stream>>>(g, d_src, e->R);
    ISB_CUDA(ctx, cudaGetLastError());
    e->last_launches += 1;
    // the validity flags and the refresh counter describe every row alike, so they stay as they are
    std::swap(e->spins, e->spins2);
    if (fields) std::swap(e->fields, e->fields2);
    if (ifields) std::swap(e->ifields, e->ifields2);
    return ISB_OK;
}

// ------------------------------------------------------------------ resampling kernels (grid: (n_pop, nb))
// flips_total += flips for every slot; with `a`, also a_r = -db E_r and the CTA maxima bmax[p*nb + b].
__global__ void __launch_bounds__(PA_THREADS) pa_weight_kernel(int P, int nb, double mdb, const double *__restrict__ E,
                                                               const unsigned long long *__restrict__ flips,
                                                               unsigned long long *flips_total, double *a, double *bmax) {
    using Reduce = cub::BlockReduce<double, PA_THREADS>;
    __shared__ typename Reduce::TempStorage tmp;
    const int p = blockIdx.x, b = blockIdx.y;
    const int i = b * PA_THREADS + threadIdx.x;
    const int64_t r = (int64_t)p * P + i;
    double v = -INFINITY;
    if (i < P) {
        flips_total[r] += flips[r];
        if (a) {
            v = __dmul_rn(mdb, E[r]);
            a[r] = v;
        }
    }
    if (!a) return;
    const double mx = Reduce(tmp).Reduce(v, MaxOp());
    if (threadIdx.x == 0) bmax[(int64_t)p * nb + b] = mx;
}

// Population max of a (from the CTA maxima), x, W, CTA-local inclusive scan of W (cloc), CTA sums bW and bx.
__global__ void __launch_bounds__(PA_THREADS) pa_scan_kernel(int P, int nb, const double *__restrict__ a,
                                                             const double *__restrict__ bmax, unsigned long long *cloc,
                                                             unsigned long long *bW, double *bx, double *pmax) {
    using ReduceD = cub::BlockReduce<double, PA_THREADS>;
    using ScanU = cub::BlockScan<unsigned long long, PA_THREADS>;
    __shared__ union {
        typename ReduceD::TempStorage red;
        typename ScanU::TempStorage scan;
    } tmp;
    __shared__ double s_max;
    const int p = blockIdx.x, b = blockIdx.y;
    const double bm = threadIdx.x < nb ? bmax[(int64_t)p * nb + threadIdx.x] : -INFINITY;
    const double mx = ReduceD(tmp.red).Reduce(bm, MaxOp());
    if (threadIdx.x == 0) {
        s_max = mx;
        if (b == 0) pmax[p] = mx;
    }
    __syncthreads();
    const int i = b * PA_THREADS + threadIdx.x;
    const int64_t r = (int64_t)p * P + i;
    double x = 0.0;
    unsigned long long w = 0;
    if (i < P) {
        // IEEE round-to-nearest; x <= 1, so x 2^32 is exact and its truncation is the floor
        x = exp(__dsub_rn(a[r], s_max));
        w = (unsigned long long)(x * 4294967296.0);
    }
    unsigned long long c, total;
    ScanU(tmp.scan).InclusiveSum(w, c, total);
    if (i < P) cloc[r] = c;
    __syncthreads();
    const double xs = ReduceD(tmp.red).Sum(x);
    if (threadIdx.x == 0) {
        bW[(int64_t)p * nb + b] = total;
        bx[(int64_t)p * nb + b] = xs;
    }
}

// Child slots j of CTA b of population p: t_j = floor((j 2^32 + U) S / (P 2^32)), parent = smallest r with C_r > t_j.
__global__ void __launch_bounds__(PA_THREADS) pa_parent_kernel(int P, int nb, uint64_t K, uint64_t seed,
                                                               const unsigned long long *__restrict__ cloc,
                                                               const unsigned long long *__restrict__ bW,
                                                               const double *__restrict__ bx,
                                                               const double *__restrict__ pmax, double *lnQ,
                                                               const int32_t *__restrict__ fam_in, int32_t *fam_out,
                                                               int32_t *parent) {
    using ScanU = cub::BlockScan<unsigned long long, PA_THREADS>;
    __shared__ typename ScanU::TempStorage tmp;
    __shared__ unsigned long long incl[PA_THREADS];   // inclusive prefix of the CTA sums of W
    const int p = blockIdx.x, b = blockIdx.y;
    const unsigned long long mine = threadIdx.x < nb ? bW[(int64_t)p * nb + threadIdx.x] : 0ull;
    unsigned long long c, S;
    ScanU(tmp).InclusiveSum(mine, c, S);
    incl[threadIdx.x] = c;
    __syncthreads();
    if (b == 0 && threadIdx.x == 0) {
        double xs = 0.0;
        for (int q = 0; q < nb; ++q) xs += bx[(int64_t)p * nb + q];
        lnQ[p] = pmax[p] + log(xs / (double)P);
    }
    const int j = b * PA_THREADS + threadIdx.x;
    if (j >= P) return;
    const uint32_t U = philox4x32_10((uint32_t)K, (uint32_t)(K >> 32), (uint32_t)p, DOM_PA_RESAMPLE << 28,
                                     (uint32_t)seed, (uint32_t)(seed >> 32)).x;
    const unsigned __int128 num = (unsigned __int128)(((uint64_t)j << 32) | U) * S;
    const unsigned long long t = (unsigned long long)(num / ((unsigned __int128)P << 32));   // t < S
    int lo = 0, hi = nb - 1;   // smallest CTA q with incl[q] > t
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (incl[mid] > t) hi = mid;
        else lo = mid + 1;
    }
    const int q = lo;
    const unsigned long long tq = t - (q ? incl[q - 1] : 0ull);   // C_r > t  <=>  cloc_r > t - (sum of the CTAs before q)
    const unsigned long long *cl = cloc + (int64_t)p * P + (int64_t)q * PA_THREADS;
    int l2 = 0, h2 = min(PA_THREADS, P - q * PA_THREADS) - 1;
    while (l2 < h2) {
        const int mid = (l2 + h2) >> 1;
        if (cl[mid] > tq) h2 = mid;
        else l2 = mid + 1;
    }
    const int64_t src = (int64_t)p * P + (int64_t)q * PA_THREADS + l2;
    const int64_t dst = (int64_t)p * P + j;
    parent[dst] = (int32_t)src;
    if (fam_in) fam_out[dst] = fam_in[src];
}

int ssf_pa_run_device(isb_ens *e, int rule, int n_pop, int64_t nT, const double *db, int64_t n_res, int64_t steps_per_T,
                      int order, int start, uint64_t seed, uint64_t step_offset, uint64_t T_offset, const PaDevice &d,
                      int *fam_final) {
    isb_model *m = e->model;
    isb_ctx *ctx = m->ctx;
    const int P = e->R / n_pop;
    const int nb = (P + PA_THREADS - 1) / PA_THREADS;
    const int64_t n = m->n, R = e->R;
    const dim3 grid(n_pop, nb);
    int cur = 0;
    for (int64_t k = 0; k < nT; ++k) {
        const int64_t t0 = k * steps_per_T;
        const int st = (int)(((int64_t)start + t0 % n) % n);
        double *Ek = d.recE ? d.recE + k * R : d.E;
        double *Mk = d.recM ? d.recM + k * R : nullptr;
        if (int rc = ssf_sweep_device(e, rule, steps_per_T, order, d.nodes, st, ISB_FLUCT_PHILOX, nullptr, seed,
                                      step_offset + (uint64_t)t0, d.T + k, steps_per_T, steps_per_T, Ek, Mk, nullptr))
            return rc;
        const bool resample = k < n_res;
        pa_weight_kernel<<<grid, PA_THREADS, 0, ctx->stream>>>(P, nb, resample ? -db[k] : 0.0, Ek, e->d_flips,
                                                               d.flips_total, resample ? d.a : nullptr, d.bmax);
        ISB_CUDA(ctx, cudaGetLastError());
        e->last_launches += 1;
        if (!resample) continue;
        pa_scan_kernel<<<grid, PA_THREADS, 0, ctx->stream>>>(P, nb, d.a, d.bmax, d.cloc, d.bW, d.bx, d.pmax);
        ISB_CUDA(ctx, cudaGetLastError());
        pa_parent_kernel<<<grid, PA_THREADS, 0, ctx->stream>>>(P, nb, T_offset + (uint64_t)k, seed, d.cloc, d.bW, d.bx,
                                                               d.pmax, d.lnQ + k * n_pop, d.fam[cur], d.fam[cur ^ 1],
                                                               d.parent);
        ISB_CUDA(ctx, cudaGetLastError());
        e->last_launches += 2;
        if (d.fam[0]) cur ^= 1;
        if (int rc = ens_select_device(e, d.parent)) return rc;
    }
    *fam_final = cur;
    return ISB_OK;
}

}  // namespace isb
