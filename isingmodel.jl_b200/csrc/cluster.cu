// cluster.cu — Swendsen-Wang cluster sweeps of sparse ensembles (isb_sw_run; the rule is documented in
// include/ising_b200.h).  One group of threads per replica for the whole call (one CTA per replica, or several replicas
// per CTA when n is small): the replica's spins (int8), its union-find labels (int32) and, when fields or cluster sizes are
// needed, one int64 word per site stay in shared memory across every sweep of the launch; the bond list (i << 16 | j, J_ij)
// and the field grid hq are read through L2 by every CTA.  Per sweep:
//   1. one Philox block per 4 bonds, the activation test of each bond (J_ij s_i s_j > 0 and u < 1 - exp(-2|J_ij|/T));
//   2. union-find in shared memory: the larger root is hooked under the smaller with atomicCAS, finds halve their paths,
//      so every label only ever moves to a smaller ancestor and the final root of a component is its smallest site;
//   3. flatten: every label becomes its root.  The walk to the root only reads, so each thread writes its own sites alone
//      and every value written is a root (a path-halving write here could land late on a site another thread has already
//      flattened and leave it pointing to a non-root);
//   4. per root: the exact int64 sum of hq_i s_i over the cluster (shared-memory atomics; skipped when h == 0);
//   5. the root's heat-bath decision P = 1 / (1 + exp(2 q S / T)), kept as the sign bit of the root's label; the sum word
//      is then reused for the cluster size (only on traced sweeps that report sum |C|^2); the flip pass.
// Nothing in the trajectory depends on the launch configuration: the labelling result (component minima) and every
// decision are functions of the sweep, replica and site indices alone.
#include <math.h>

#include <algorithm>
#include <vector>

#include "common.cuh"
#include "handles.hpp"

namespace isb {

constexpr int SW_THREADS_MAX = 512;

struct SwParams {
    const uint32_t *pair;   // [nbonds] i << 16 | j
    const double *J;        // [nbonds]
    const int32_t *hq;      // [n] fields on the grid
    const double *h;        // [n] the model's fields (traced energies)
    int8_t *spins;
    int64_t lds;
    int n, R;
    int64_t nbonds;
    bool has_h, need_sum;
    double q2;              // 2 q
    int64_t nsweeps;
    uint64_t seed, sweep_offset;
    const double *Tsched;
    const double *tscale;
    int64_t sweeps_per_T, trace_every;
    double *out_E, *out_M;
    int64_t *out_csq;
    unsigned long long *flips;
    int tpr;                // threads per replica (a multiple of 32)
    int rpc;                // replicas per CTA
    size_t smem_per_rep;    // bytes of dynamic shared memory per replica (a multiple of 16)
};

// Root of x.  Path halving: a write replaces the parent of a non-root by its grandparent, so a label only ever moves to an
// ancestor (never to a larger index, never onto a root), whatever the other threads do at the same time.
__device__ __forceinline__ int sw_find(volatile int32_t *lab, int x) {
    while (true) {
        const int p = lab[x];
        if (p == x) return x;
        const int g = lab[p];
        if (g == p) return p;
        lab[x] = g;
        x = g;
    }
}

// Join the components of a and b: the larger root is hooked under the smaller one.
__device__ __forceinline__ void sw_union(int32_t *lab, int a, int b) {
    volatile int32_t *vl = lab;
    while (true) {
        a = sw_find(vl, a);
        b = sw_find(vl, b);
        if (a == b) return;
        if (a > b) {
            const int t = a;
            a = b;
            b = t;
        }
        const int old = atomicCAS(&lab[b], b, a);
        if (old == b) return;
        b = old;   // b was hooked meanwhile: continue from its new parent
    }
}

// Root of x without writing anything (the flatten pass).
__device__ __forceinline__ int sw_root(const volatile int32_t *lab, int x) {
    int p;
    while ((p = lab[x]) != x) x = p;
    return x;
}

__device__ __forceinline__ long long warp_sum_ll(long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ double sw_uniform(uint32_t w) { return ((double)w + 0.5) * 2.3283064365386963e-10; }

// (80 registers without spills: three CTAs of 256 threads per SM)
__global__ void __maxnreg__(80) sw_kernel(const SwParams p) {
    extern __shared__ __align__(16) unsigned char sm_raw[];
    __shared__ double red_d[SW_THREADS_MAX / 32];
    __shared__ long long red_m[SW_THREADS_MAX / 32], red_c[SW_THREADS_MAX / 32];
    // group g of the CTA runs replica r; a group past the last replica keeps n = 0 and only joins the barriers
    const int g = threadIdx.x / p.tpr, tid = threadIdx.x % p.tpr, nt = p.tpr, wbase = g * (p.tpr / 32);
    const int r = blockIdx.x * p.rpc + g;
    const bool live = r < p.R;
    const int n = live ? p.n : 0;
    const int64_t nbonds = live ? p.nbonds : 0;
    unsigned char *base = sm_raw + (size_t)g * p.smem_per_rep;
    long long *sum = reinterpret_cast<long long *>(base);                                           // [n] if need_sum
    int32_t *lab = reinterpret_cast<int32_t *>(base + (p.need_sum ? 8 * (size_t)p.n : 0));          // [n]
    int8_t *sp = reinterpret_cast<int8_t *>(lab + p.n);                                             // [n]
    int8_t *gs = p.spins + (int64_t)r * p.lds;
    for (int i = tid; i < n; i += nt) sp[i] = gs[i];
    const uint32_t k0 = (uint32_t)p.seed, k1 = (uint32_t)(p.seed >> 32);
    const double tsc = (live && p.tscale) ? __ldg(&p.tscale[r]) : 1.0;
    const int64_t nquads = (nbonds + 3) >> 2;
    unsigned long long nflips = 0;
    double memo_aJ = -1.0, memo_T = 0.0, memo_p = 0.0;   // the last bond threshold this thread computed
    int64_t trace_idx = 0;
    __syncthreads();
    for (int64_t k = 0; k < p.nsweeps; ++k) {
        const uint64_t Ka = p.sweep_offset + (uint64_t)k;
        const uint32_t c0 = (uint32_t)Ka, c1 = (uint32_t)(Ka >> 32);
        const double T = __dmul_rn(__ldg(&p.Tsched[k / p.sweeps_per_T]), tsc);
        for (int i = tid; i < n; i += nt) {
            lab[i] = i;
            if (p.need_sum) sum[i] = 0;
        }
        __syncthreads();
        // 1-2. bonds
        for (int64_t qd = tid; qd < nquads; qd += nt) {
            const Philox4 w = philox4x32_10(c0, c1, (uint32_t)r, (DOM_SW_BOND << 28) | (uint32_t)qd, k0, k1);
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const int64_t e = qd * 4 + c;
                if (e >= nbonds) break;
                const uint32_t pr = __ldg(&p.pair[e]);
                const int i = (int)(pr >> 16), j = (int)(pr & 0xffffu);
                const double J = __ldg(&p.J[e]);
                if ((J > 0.0) != (sp[i] == sp[j])) continue;   // J s_i s_j < 0: never active
                const double aJ = fabs(J);
                if (aJ != memo_aJ || T != memo_T) {
                    memo_aJ = aJ;
                    memo_T = T;
                    memo_p = __dsub_rn(1.0, exp(__ddiv_rn(-2.0 * aJ, T)));
                }
                if (sw_uniform(philox_pick(w, (uint32_t)c)) < memo_p) sw_union(lab, i, j);
            }
        }
        __syncthreads();
        // 3. flatten
        for (int i = tid; i < n; i += nt) lab[i] = sw_root(lab, i);
        __syncthreads();
        // 4. cluster field sums (exact integers)
        if (p.has_h) {
            for (int i = tid; i < n; i += nt) {
                const int hv = __ldg(&p.hq[i]);
                if (hv) atomicAdd(reinterpret_cast<unsigned long long *>(&sum[lab[i]]),
                                  (unsigned long long)(long long)(sp[i] > 0 ? hv : -hv));
            }
            __syncthreads();
        }
        // 5. one heat-bath decision per root, kept as the sign bit of its label
        for (int i = tid; i < n; i += nt) {
            if (lab[i] != i) continue;
            double P = 0.5;   // what the formula gives for S = 0 (exp(0) = 1)
            if (p.has_h) {
                const double x = __ddiv_rn(__dmul_rn(p.q2, (double)sum[i]), T);
                P = __ddiv_rn(1.0, __dadd_rn(1.0, exp(x)));
            }
            if (p.need_sum) sum[i] = 0;   // the word counts the cluster's sites from here on
            const Philox4 z = philox4x32_10(c0, c1, (uint32_t)r, (DOM_SW_FLIP << 28) | (uint32_t)(i >> 2), k0, k1);
            if (sw_uniform(philox_pick(z, (uint32_t)(i & 3))) < P) lab[i] = (int32_t)((uint32_t)i | 0x80000000u);
        }
        __syncthreads();
        const bool trace = p.trace_every > 0 && (k + 1) % p.trace_every == 0;
        const bool sizes = trace && p.out_csq;
        if (sizes) {
            for (int i = tid; i < n; i += nt) atomicAdd(reinterpret_cast<unsigned long long *>(&sum[lab[i] & 0x7fffffff]), 1ull);
            __syncthreads();
        }
        // flips (and the magnetisation / sum of |C|^2 of a traced sweep)
        long long mag = 0, csq = 0;
        for (int i = tid; i < n; i += nt) {
            const int root = lab[i] & 0x7fffffff;
            int8_t s = sp[i];
            if (lab[root] < 0) {
                s = (int8_t)-s;
                sp[i] = s;
                ++nflips;
            }
            mag += s;
            if (sizes && root == i) csq += sum[i] * sum[i];
        }
        if (trace) {
            __syncthreads();   // every flip is in
            double ev = 0.0;
            for (int64_t e = tid; e < nbonds; e += nt) {
                const uint32_t pr = __ldg(&p.pair[e]);
                const double J = __ldg(&p.J[e]);
                ev -= sp[pr >> 16] == sp[pr & 0xffffu] ? J : -J;
            }
            for (int i = tid; i < n; i += nt) {
                const double hv = __ldg(&p.h[i]);
                ev -= sp[i] > 0 ? hv : -hv;
            }
            ev = warp_sum(ev);
            mag = warp_sum_ll(mag);
            csq = warp_sum_ll(csq);
            const int wid = threadIdx.x >> 5;
            if ((tid & 31) == 0) {
                red_d[wid] = ev;
                red_m[wid] = mag;
                red_c[wid] = csq;
            }
            __syncthreads();
            if (tid == 0 && live) {
                for (int q = 1; q < nt / 32; ++q) {
                    ev += red_d[wbase + q];
                    mag += red_m[wbase + q];
                    csq += red_c[wbase + q];
                }
                const int64_t o = trace_idx * p.R + r;
                if (p.out_E) p.out_E[o] = ev;
                if (p.out_M) p.out_M[o] = (double)mag;
                if (p.out_csq) p.out_csq[o] = csq;
            }
            ++trace_idx;
        }
        __syncthreads();   // labels, sums and the reduction words are rewritten by the next sweep
    }
    for (int i = tid; i < n; i += nt) gs[i] = sp[i];
    const long long fl = warp_sum_ll((long long)nflips);
    if ((tid & 31) == 0) red_m[threadIdx.x >> 5] = fl;
    __syncthreads();
    if (tid == 0 && live) {
        long long tot = 0;
        for (int q = 0; q < nt / 32; ++q) tot += red_m[wbase + q];
        p.flips[r] = (unsigned long long)tot;
    }
}

// ------------------------------------------------------------------ host
int sw_model_prepare(isb_model *m) {
    isb_ctx *ctx = m->ctx;
    SparseModel *sm = (SparseModel *)m->sp;
    if (sm->sw_ready) return ISB_OK;
    const int n = m->n;
    std::vector<int> rowptr((size_t)n + 1), col((size_t)sm->nnz);
    std::vector<double> val((size_t)sm->nnz), h((size_t)n);
    ISB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ISB_CUDA(ctx, cudaMemcpy(rowptr.data(), sm->rowptr, rowptr.size() * sizeof(int), cudaMemcpyDeviceToHost));
    if (sm->nnz) {
        ISB_CUDA(ctx, cudaMemcpy(col.data(), sm->col, col.size() * sizeof(int), cudaMemcpyDeviceToHost));
        ISB_CUDA(ctx, cudaMemcpy(val.data(), sm->val, val.size() * sizeof(double), cudaMemcpyDeviceToHost));
    }
    ISB_CUDA(ctx, cudaMemcpy(h.data(), m->h64, h.size() * sizeof(double), cudaMemcpyDeviceToHost));
    // bonds: row i of the CSR (columns ascending), columns > i, rows ascending
    std::vector<uint32_t> pair;
    std::vector<double> J;
    for (int i = 0; i < n; ++i)
        for (int e = rowptr[i]; e < rowptr[i + 1]; ++e)
            if (col[e] > i) {
                pair.push_back(((uint32_t)i << 16) | (uint32_t)col[e]);
                J.push_back(val[e]);
            }
    // fields on the grid q = 2^(e_h - 30), e_h the smallest integer with max|h| <= 2^e_h: |hq_i| <= 2^30
    double hmax = 0.0;
    for (double v : h) hmax = std::max(hmax, std::fabs(v));
    std::vector<int32_t> hq((size_t)n, 0);
    double q = 1.0;
    if (hmax > 0.0) {
        int ex = 0;
        const double f = std::frexp(hmax, &ex);   // hmax = f 2^ex, f in [0.5, 1)
        const int eh = f == 0.5 ? ex - 1 : ex;
        q = std::ldexp(1.0, eh - 30);
        for (int i = 0; i < n; ++i) hq[i] = (int32_t)std::nearbyint(h[i] / q);
    }
    // allocate and fill into locals; the model takes them only once everything has succeeded
    const size_t nb = std::max<size_t>(pair.size(), 1);
    uint32_t *d_pair = nullptr;
    double *d_J = nullptr;
    int32_t *d_hq = nullptr;
    cudaError_t ce = cudaMalloc(&d_pair, nb * sizeof(uint32_t));
    if (ce == cudaSuccess) ce = cudaMalloc(&d_J, nb * sizeof(double));
    if (ce == cudaSuccess) ce = cudaMalloc(&d_hq, (size_t)n * sizeof(int32_t));
    if (ce == cudaSuccess && !pair.empty()) {
        ce = cudaMemcpy(d_pair, pair.data(), pair.size() * sizeof(uint32_t), cudaMemcpyHostToDevice);
        if (ce == cudaSuccess) ce = cudaMemcpy(d_J, J.data(), J.size() * sizeof(double), cudaMemcpyHostToDevice);
    }
    if (ce == cudaSuccess) ce = cudaMemcpy(d_hq, hq.data(), hq.size() * sizeof(int32_t), cudaMemcpyHostToDevice);
    if (ce != cudaSuccess) {
        cudaFree(d_pair);
        cudaFree(d_J);
        cudaFree(d_hq);
        return fail(ctx, ISB_ERR_CUDA, "isb_sw_run: uploading the bond list failed: %s", cudaGetErrorString(ce));
    }
    sm->sw_pair = d_pair;
    sm->sw_J = d_J;
    sm->sw_hq = d_hq;
    sm->sw_nbonds = (int64_t)pair.size();
    sm->sw_q = q;
    sm->sw_has_h = hmax > 0.0;
    sm->sw_ready = true;
    return ISB_OK;
}

void sw_model_free(SparseModel *sm) {
    cudaFree(sm->sw_pair);
    cudaFree(sm->sw_J);
    cudaFree(sm->sw_hq);
    sm->sw_pair = nullptr;
    sm->sw_J = nullptr;
    sm->sw_hq = nullptr;
    sm->sw_ready = false;
}

int sw_run_device(isb_ens *e, int64_t nsweeps, uint64_t seed, uint64_t sweep_offset, const double *d_T,
                  int64_t sweeps_per_T, int64_t trace_every, double *d_E, double *d_M, int64_t *d_csq) {
    isb_model *m = e->model;
    isb_ctx *ctx = m->ctx;
    SparseModel *sm = (SparseModel *)m->sp;
    if (nsweeps <= 0) return ISB_OK;
    const int n = m->n;
    SwParams p{};
    p.pair = sm->sw_pair;
    p.J = sm->sw_J;
    p.hq = sm->sw_hq;
    p.h = m->h64;
    p.spins = e->spins;
    p.lds = e->lds;
    p.n = n;
    p.R = e->R;
    p.nbonds = sm->sw_nbonds;
    p.has_h = sm->sw_has_h;
    p.need_sum = sm->sw_has_h || d_csq != nullptr;
    p.q2 = 2.0 * sm->sw_q;
    p.nsweeps = nsweeps;
    p.seed = seed;
    p.sweep_offset = sweep_offset;
    p.Tsched = d_T;
    p.tscale = e->d_tscale;
    p.sweeps_per_T = sweeps_per_T;
    p.trace_every = (d_E || d_M || d_csq) ? trace_every : 0;
    p.out_E = d_E;
    p.out_M = d_M;
    p.out_csq = d_csq;
    p.flips = e->d_flips;
    // about four sites per thread, 32 .. 512 threads per replica, and replicas of fewer than 256 threads packed into CTAs
    // of 256: a function of n alone (the trajectory does not depend on it; the summation order of traced E does)
    p.tpr = std::min(SW_THREADS_MAX, std::max(32, ((n + 3) / 4 + 31) / 32 * 32));
    p.rpc = std::max(1, std::min(256 / p.tpr, e->R));
    p.smem_per_rep = ((p.need_sum ? 8 * (size_t)n : 0) + 5 * (size_t)n + 15) / 16 * 16;
    const size_t smem = p.smem_per_rep * (size_t)p.rpc;
    if (smem + 1024 > ctx->smem_optin)   // (and the kernel's static reduction words)
        return fail(ctx, ISB_ERR_UNSUPPORTED, "isb_sw_run: %zu bytes of shared memory per replica exceed the %zu of this device",
                    smem, ctx->smem_optin);
    const int grid = (e->R + p.rpc - 1) / p.rpc;
    cudaError_t ce = cudaFuncSetAttribute(sw_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (ce == cudaSuccess) {
        sw_kernel<<<grid, p.tpr * p.rpc, smem, ctx->stream>>>(p);
        ce = cudaGetLastError();
    }
    if (ce != cudaSuccess) return fail(ctx, ISB_ERR_CUDA, "sw_kernel launch failed: %s", cudaGetErrorString(ce));
    e->last_launches += 1;
    return ISB_OK;
}

}  // namespace isb
