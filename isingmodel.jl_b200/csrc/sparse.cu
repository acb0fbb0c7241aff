// sparse.cu — single-spin-flip sweeps for SPARSE couplings (SURVEY §8f rank 1).
//
// The reference's own tests and demo build their SpinSystem from a SparseMatrixCSC (test/runtests.jl:20,
// demo.jl:60-62); a 32x32 lattice stored densely wastes 256x the bandwidth.  Same rules and the same step loop
// as K1 (src/SingleSpinFlip.jl:31-36,46-55,65-74; src/SamplingHelper.jl:45-49), different data layout:
//   * J as CSR rows (J is symmetric, so row i == column i of the caller's CSC), values in double;
//   * one warp per chain, the chain's local fields in SHARED memory (double[n]) and its spins as bytes next to
//     them; an accepted flip of site i touches only the deg(i) neighbours: fld[j] += +-2 J_ij;
//   * sequential sweeps use the same 32-site speculation as K1 (all lanes decide at once, the first flipping
//     lane is applied, later lanes re-read their field and decide again).
// Decisions in double with the reference's operation order; ties give +1 (src/SpinSystems.jl:163-171).
#include <stdlib.h>

#include <algorithm>
#include <vector>

#include "common.cuh"
#include "handles.hpp"

namespace isb {

struct SparseModel {
    int64_t nnz = 0;
    int *rowptr = nullptr;   // [n+1]
    int *col = nullptr;      // [nnz] ascending within a row
    double *val = nullptr;   // [nnz]
    int maxdeg = 0;
    void *lattice = nullptr;  // periodic square lattice recognised: sequential sweeps run in lattice.cu
    std::vector<double> ars;  // row sums of |J| (near-tie guard, completed with |h| by the caller)
    std::vector<double> vals;
};

struct SpParams {
    const int *rowptr;
    const int *col;
    const double *val;
    const double *hext;
    int8_t *spins;
    int64_t lds;
    double *fields;  // [R][npad]
    int n, npad, R, rule;
    double ecoef;
    int64_t nsteps;
    int start;
    const int32_t *nodes;
    int fluct_mode;
    const double *fluct;
    uint64_t seed, step_offset;
    const double *Tsched;
    const double *tscale;
    int64_t steps_per_T;
    int64_t trace_every;
    double *out_E, *out_M;
    int8_t *out_S;
    int64_t ldS;
    unsigned long long *flips, *near_ties;
    double tie_eps;
    int chains_per_cta;
    double guard;   // near-tie guard (see SsfParams::guard): 0 = arithmetic exact, no guard
    double hsign;
};

// GLOBALF: the chain's fields and spins stay in global memory (models too large for 9 N bytes of shared memory per
// chain: the reference has no size limit); same code, the working set is served by L1 / L2.
template <bool LIST, bool GLOBALF = false>
__global__ void ssf_sparse_kernel(const SpParams p) {
    extern __shared__ __align__(16) unsigned char sm_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int r = blockIdx.x * p.chains_per_cta + warp;
    if (r >= p.R) return;
    const size_t per_chain = (size_t)p.npad * sizeof(double) + (size_t)p.npad;
    double *fld = GLOBALF ? p.fields + (int64_t)r * p.npad : reinterpret_cast<double *>(sm_raw + (size_t)warp * per_chain);
    int8_t *sp = GLOBALF ? p.spins + (int64_t)r * p.lds : reinterpret_cast<int8_t *>(fld + p.npad);
    constexpr uint32_t FULL = 0xffffffffu;
    if constexpr (!GLOBALF) {
        for (int i = lane; i < p.npad; i += 32) {
            fld[i] = p.fields[(int64_t)r * p.npad + i];
            sp[i] = i < p.n ? p.spins[(int64_t)r * p.lds + i] : (int8_t)1;
        }
    }
    __syncwarp();
    const int rule = p.rule;
    const bool metro = rule == 2, audit = p.tie_eps > 0.0;
    const double tsc = p.tscale ? __ldg(&p.tscale[r]) : 1.0;
    unsigned long long nflips = 0, nties = 0;

    // fld[j] += d * J[i][j] over the neighbours of site i (distinct j: no conflicts), spin flipped by lane 0
    auto apply_flip = [&](int i, bool up) {
        const double d = up ? 2.0 : -2.0;
        const int a = __ldg(&p.rowptr[i]), b = __ldg(&p.rowptr[i + 1]);
        for (int e = a + lane; e < b; e += 32) fld[__ldg(&p.col[e])] += d * __ldg(&p.val[e]);
        if (lane == 0) sp[i] = up ? (int8_t)1 : (int8_t)-1;
        __syncwarp();
    };
    // the reference's fresh field of site i: stored neighbours in ascending index (the skipped terms are +-0), then +- h_i
    auto exact_field = [&](int i) -> double {
        double acc = 0.0;
        for (int e = __ldg(&p.rowptr[i]); e < __ldg(&p.rowptr[i + 1]); ++e) {
            const double v = __ldg(&p.val[e]);
            acc = __dadd_rn(acc, sp[__ldg(&p.col[e])] > 0 ? v : -v);
        }
        return __dadd_rn(acc, p.hsign * __ldg(&p.hext[i]));
    };
    auto fluct_at = [&](int64_t tl) -> double {
        if (rule == 0) return 0.0;
        if (p.fluct_mode == ISB_FLUCT_PHILOX)
            return ssf_fluct_from_word(rule, philox_step_word(p.seed, DOM_SSF_FLUCT, (uint32_t)r, p.step_offset + (uint64_t)tl));
        return p.fluct_mode == ISB_FLUCT_SHARED ? __ldg(&p.fluct[tl]) : __ldg(&p.fluct[(int64_t)r * p.nsteps + tl]);
    };
    auto write_trace = [&](int64_t idx) {
        double sf = 0.0, sh = 0.0;
        int m = 0;
        for (int i = lane; i < p.n; i += 32) {
            const bool up = sp[i] > 0;
            sf += up ? fld[i] : -fld[i];
            const double hv = __ldg(&p.hext[i]);
            sh += up ? hv : -hv;
            m += up ? 1 : -1;
        }
        sf = warp_sum(sf);
        sh = warp_sum(sh);
        m = warp_sum_int(m);
        if (lane == 0) {
            if (p.out_E) p.out_E[idx * p.R + r] = -0.5 * sf - p.ecoef * sh;
            if (p.out_M) p.out_M[idx * p.R + r] = (double)m;
        }
        if (p.out_S)
            for (int i = lane; i < p.n; i += 32) p.out_S[(idx * p.R + r) * p.ldS + i] = sp[i];
    };
    int64_t next_trace = p.trace_every > 0 ? p.trace_every : INT64_MAX, trace_idx = 0;

    if constexpr (!LIST) {
        int64_t t = 0;
        int site = p.start;
        while (t < p.nsteps) {
            int len = 32;
            if (p.n - site < len) len = p.n - site;
            if (p.nsteps - t < len) len = (int)(p.nsteps - t);
            if (next_trace - t < len) len = (int)(next_trace - t);
            const bool mine = lane < len;
            const int64_t tl = t + lane;
            const double Tl = mine ? __dmul_rn(__ldg(&p.Tsched[tl / p.steps_per_T]), tsc) : 0.0;
            const double ftl = __dmul_rn(mine ? fluct_at(tl) : 0.0, Tl);
            const int i = site + (mine ? lane : 0);
            bool mybit = sp[i] > 0;
            uint32_t rem = __ballot_sync(FULL, mine);
            while (true) {
                double h2 = 2.0 * fld[i];
                const double fts = metro ? (mybit ? ftl : -ftl) : ftl;
                double x = __dsub_rn(h2, fts);
                if (p.guard > 0.0 && fabs(x) < p.guard && ((rem >> lane) & 1u)) {   // rare: decide on the fresh row dot
                    const double ex = exact_field(i);
                    fld[i] = ex;
                    h2 = 2.0 * ex;
                    x = __dsub_rn(h2, fts);
                }
                const bool nb = !(x < 0.0);
                const uint32_t fm = __ballot_sync(FULL, nb != mybit) & rem;
                if (audit) {
                    const uint32_t tm = __ballot_sync(FULL, fabs(x) < p.tie_eps) & rem;
                    nties += __popc(fm ? (tm & ((2u << (__ffs(fm) - 1)) - 1u)) : tm);
                }
                if (fm == 0) break;
                const int l0 = __ffs(fm) - 1;
                const bool up = (__ballot_sync(FULL, nb) >> l0) & 1u;
                apply_flip(site + l0, up);
                if (lane == l0) mybit = up;
                ++nflips;
                rem &= ~((2u << l0) - 1u);
                if (rem == 0) break;
            }
            t += len;
            site += len;
            if (site >= p.n) site = 0;
            if (t == next_trace) {
                write_trace(trace_idx++);
                next_trace += p.trace_every;
            }
        }
    } else {
        for (int64_t t = 0; t < p.nsteps; ++t) {
            const int i = __ldg(&p.nodes[t]);
            const double T = __dmul_rn(__ldg(&p.Tsched[t / p.steps_per_T]), tsc);
            const double ft = __dmul_rn(fluct_at(t), T);
            const bool mybit = sp[i] > 0;
            double x = __dsub_rn(2.0 * fld[i], metro ? (mybit ? ft : -ft) : ft);
            if (p.guard > 0.0 && fabs(x) < p.guard) {
                const double ex = exact_field(i);
                __syncwarp();
                if (lane == 0) fld[i] = ex;
                __syncwarp();
                x = __dsub_rn(2.0 * ex, metro ? (mybit ? ft : -ft) : ft);
            }
            const bool nb = !(x < 0.0);
            if (audit && fabs(x) < p.tie_eps) ++nties;
            if (nb != mybit) {
                apply_flip(i, nb);
                ++nflips;
            }
            if (t + 1 == next_trace) {
                write_trace(trace_idx++);
                next_trace += p.trace_every;
            }
        }
    }
    __syncwarp();
    if constexpr (!GLOBALF) {
        for (int i = lane; i < p.npad; i += 32) {
            p.fields[(int64_t)r * p.npad + i] = fld[i];
            if (i < p.n) p.spins[(int64_t)r * p.lds + i] = sp[i];
        }
    }
    if (lane == 0) {
        p.flips[r] = nflips;
        if (nties) atomicAdd(p.near_ties, nties);
    }
}

// g_i = sum_j J_ij s_j over the stored entries in ascending j (bit-identical to the dense sequential sum:
// the skipped terms are +-0), then + / - h_i.
__global__ void sparse_field_kernel(const int *rowptr, const int *col, const double *val, const double *h,
                                    const int8_t *spins, int64_t lds, double *out, int64_t ldo, int n, int nout, int R,
                                    double hsign) {
    const int64_t total = (int64_t)R * nout;
    for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = idx / nout;
        const int i = (int)(idx % nout);
        double v = 0.0;
        if (i < n) {
            double acc = 0.0;
            for (int e = rowptr[i]; e < rowptr[i + 1]; ++e) acc += val[e] * (double)spins[r * lds + col[e]];
            v = hsign > 0 ? acc + h[i] : acc - h[i];
        }
        out[r * ldo + i] = v;
    }
}

// E_r = -1/2 sum_i s_i g_i - sum_i h_i s_i ; one warp per replica
__global__ void sparse_energy_kernel(const int *rowptr, const int *col, const double *val, const double *h,
                                     const int8_t *spins, int64_t lds, double *E, int n, int R) {
    const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (r >= R) return;
    double q = 0.0, l = 0.0;
    for (int i = lane; i < n; i += 32) {
        double acc = 0.0;
        for (int e = rowptr[i]; e < rowptr[i + 1]; ++e) acc += val[e] * (double)spins[(int64_t)r * lds + col[e]];
        const double si = (double)spins[(int64_t)r * lds + i];
        q += si * acc;
        l += h[i] * si;
    }
    q = warp_sum(q);
    l = warp_sum(l);
    if (lane == 0) E[r] = -0.5 * q - l;
}

// ------------------------------------------------------------------ host
int sparse_model_init(isb_model *m, int n, const int64_t *colptr, const int32_t *rowval, const double *nzval, int *warn) {
    isb_ctx *ctx = m->ctx;
    // symmetrise by the upper triangle when needed and drop the diagonal (src/SpinSystems.jl:31-38)
    std::vector<std::vector<std::pair<int, double>>> rows((size_t)n);
    bool diag = false;
    // upper triangle entries (i <= j) of column j, and the lower ones for the symmetry check
    std::vector<std::vector<std::pair<int, double>>> upper((size_t)n), lower((size_t)n);
    for (int j = 0; j < n; ++j)
        for (int64_t e = colptr[j]; e < colptr[j + 1]; ++e) {
            const int i = rowval[e];
            const double v = nzval[e];
            if (i < 0 || i >= n) return fail(ctx, ISB_ERR_ARG, "isb_model_sparse: row index %d outside [0, %d)", i, n);
            if (!std::isfinite(v)) return fail(ctx, ISB_ERR_NONFINITE, "isb_model_sparse: J[%d,%d] is not finite", i, j);
            if (i == j) {
                if (v != 0.0) diag = true;
            } else if (i < j) {
                if (v != 0.0) upper[j].push_back({i, v});  // element (i, j), i < j
            } else {
                if (v != 0.0) lower[i].push_back({j, v});  // element (i, j), i > j stored under row i as (j)
            }
        }
    bool sym = true;
    for (int j = 0; j < n && sym; ++j) {
        auto a = upper[j], b = lower[j];  // (i, J_ij) for i < j   vs   (i, J_ji) for i < j
        std::sort(a.begin(), a.end());
        std::sort(b.begin(), b.end());
        sym = a == b;
    }
    for (int j = 0; j < n; ++j)
        for (auto &pr : upper[j]) {
            rows[pr.first].push_back({j, pr.second});
            rows[j].push_back({pr.first, pr.second});
        }
    if (warn) *warn = (sym ? 0 : 1) | (diag ? 2 : 0);
    SparseModel *sm = new SparseModel();
    m->sp = sm;
    std::vector<int> rowptr((size_t)n + 1, 0), col;
    std::vector<double> val;
    for (int i = 0; i < n; ++i) {
        std::sort(rows[i].begin(), rows[i].end());
        for (auto &pr : rows[i]) {
            col.push_back(pr.first);
            val.push_back(pr.second);
        }
        rowptr[i + 1] = (int)col.size();
        sm->maxdeg = std::max(sm->maxdeg, rowptr[i + 1] - rowptr[i]);
    }
    sm->nnz = (int64_t)col.size();
    sm->lattice = lattice_detect(ctx, n, rows);
    {
        std::vector<double> ars((size_t)n, 0.0);
        for (int i = 0; i < n; ++i)
            for (int e = rowptr[i]; e < rowptr[i + 1]; ++e) ars[i] += fabs(val[e]);
        sm->ars = ars;
        sm->vals = val;
    }
    const size_t nz = std::max<size_t>(col.size(), 1);
    ISB_CUDA(ctx, cudaMalloc(&sm->rowptr, (n + 1) * sizeof(int)));
    ISB_CUDA(ctx, cudaMalloc(&sm->col, nz * sizeof(int)));
    ISB_CUDA(ctx, cudaMalloc(&sm->val, nz * sizeof(double)));
    ISB_CUDA(ctx, cudaMemcpy(sm->rowptr, rowptr.data(), (n + 1) * sizeof(int), cudaMemcpyHostToDevice));
    if (!col.empty()) {
        ISB_CUDA(ctx, cudaMemcpy(sm->col, col.data(), col.size() * sizeof(int), cudaMemcpyHostToDevice));
        ISB_CUDA(ctx, cudaMemcpy(sm->val, val.data(), val.size() * sizeof(double), cudaMemcpyHostToDevice));
    }
    return ISB_OK;
}

void sparse_model_set_guard(isb_model *m, const double *h_host) {
    SparseModel *sm = (SparseModel *)m->sp;
    std::vector<double> ars = sm->ars;
    for (int i = 0; i < m->n; ++i) ars[i] += fabs(h_host[i]);
    m->guard = ssf_guard_from(ars.data(), sm->vals.data(), sm->vals.size(), h_host, m->n);
    sm->ars.clear();
    sm->vals.clear();
}

bool sparse_model_lattice(const isb_model *m) { return m->sp && ((const SparseModel *)m->sp)->lattice; }

void sparse_model_free(isb_model *m) {
    SparseModel *sm = (SparseModel *)m->sp;
    if (!sm) return;
    cudaFree(sm->rowptr);
    cudaFree(sm->col);
    cudaFree(sm->val);
    lattice_free(sm->lattice);
    delete sm;
    m->sp = nullptr;
}

int sparse_field_device(isb_ens *e, double *d_out, int64_t ld, int nout, double hsign) {
    isb_model *m = e->model;
    SparseModel *sm = (SparseModel *)m->sp;
    sparse_field_kernel<<<m->ctx->num_sms * 8, 256, 0, m->ctx->stream>>>(sm->rowptr, sm->col, sm->val, m->h64, e->spins,
                                                                         e->lds, d_out, ld, m->n, nout, e->R, hsign);
    ISB_CUDA(m->ctx, cudaGetLastError());
    return ISB_OK;
}

int sparse_energy_device(isb_ens *e, double *d_E) {
    isb_model *m = e->model;
    SparseModel *sm = (SparseModel *)m->sp;
    sparse_energy_kernel<<<(e->R + 7) / 8, 256, 0, m->ctx->stream>>>(sm->rowptr, sm->col, sm->val, m->h64, e->spins, e->lds,
                                                                     d_E, m->n, e->R);
    ISB_CUDA(m->ctx, cudaGetLastError());
    return ISB_OK;
}

int ssf_sparse_run_device(isb_ens *e, int rule, int64_t nsteps, int order, const int32_t *d_nodes, int start,
                          int fluct_mode, const double *d_fluct, uint64_t seed, uint64_t step_offset, const double *d_T,
                          int64_t steps_per_T, int64_t trace_every, double *d_E, double *d_M, int8_t *d_S) {
    isb_model *m = e->model;
    isb_ctx *ctx = m->ctx;
    SparseModel *sm = (SparseModel *)m->sp;
    if (nsteps <= 0) return ISB_OK;
    // (ISB_ORDER_CHECKERBOARD arrives on lattices only: the entry points refuse it elsewhere, see sparse_model_lattice)
    if (sm->lattice && (order == ISB_ORDER_SEQUENTIAL || order == ISB_ORDER_CHECKERBOARD))
        return ssf_lattice_run_device(e, sm->lattice, rule, nsteps, order, start, fluct_mode, d_fluct, seed, step_offset, d_T,
                                      steps_per_T, trace_every, d_E, d_M, d_S);
    const int sign = rule == ISB_RULE_HOPFIELD ? -1 : +1;
    if (e->steps_since_refresh >= (int64_t)ISB_FIELD_REFRESH_SWEEPS * m->n) e->fields_rule_sign = 0;  // bound the drift
    if (e->fields_rule_sign != sign) {
        int rc = sparse_field_device(e, (double *)e->fields, m->npad, m->npad, (double)sign);
        if (rc) return rc;
        e->fields_rule_sign = sign;
        e->steps_since_refresh = 0;
        e->last_launches += 1;
    }
    e->steps_since_refresh += nsteps;
    const size_t per_chain = (size_t)m->npad * 9;
    int chains = (int)std::min<size_t>(24, (ctx->smem_optin - 1024) / per_chain);
    // N above ~25 000 sites: 9 N bytes per chain no longer fit the shared memory; the chain's fields and spins then stay
    // in global memory (ISB_SPARSE_GLOBAL=1 forces this variant, for tests)
    bool globalf = chains < 1;
    if (const char *env = getenv("ISB_SPARSE_GLOBAL")) globalf = globalf || atoi(env) != 0;
    if (globalf) chains = 8;
    // spread the chains over the SMs first (one warp = one chain)
    const int per_sm = (e->R + ctx->num_sms - 1) / ctx->num_sms;
    chains = std::max(1, std::min(chains, per_sm));
    const int grid = (e->R + chains - 1) / chains;
    SpParams p{};
    p.rowptr = sm->rowptr; p.col = sm->col; p.val = sm->val; p.hext = m->h64;
    p.spins = e->spins; p.lds = e->lds; p.fields = (double *)e->fields;
    p.n = m->n; p.npad = m->npad; p.R = e->R; p.rule = rule;
    p.ecoef = rule == ISB_RULE_HOPFIELD ? 1.5 : 0.5;
    p.nsteps = nsteps; p.start = start; p.nodes = d_nodes;
    p.fluct_mode = fluct_mode; p.fluct = d_fluct; p.seed = seed; p.step_offset = step_offset;
    p.Tsched = d_T; p.tscale = e->d_tscale; p.steps_per_T = steps_per_T; p.trace_every = trace_every;
    p.out_E = d_E; p.out_M = d_M; p.out_S = d_S; p.ldS = m->n; p.flips = e->d_flips; p.near_ties = e->d_counters; p.tie_eps = e->tie_eps;
    p.chains_per_cta = chains;
    p.guard = m->guard;
    p.hsign = rule == ISB_RULE_HOPFIELD ? -1.0 : 1.0;
    const size_t smem = globalf ? 0 : per_chain * chains;
    cudaError_t ce = cudaSuccess;
    if (globalf) {
        if (order != ISB_ORDER_SEQUENTIAL)
            ssf_sparse_kernel<true, true><<<grid, 32 * chains, 0, ctx->stream>>>(p);
        else
            ssf_sparse_kernel<false, true><<<grid, 32 * chains, 0, ctx->stream>>>(p);
    } else if (order != ISB_ORDER_SEQUENTIAL) {
        ce = cudaFuncSetAttribute(ssf_sparse_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (ce == cudaSuccess) ssf_sparse_kernel<true><<<grid, 32 * chains, smem, ctx->stream>>>(p);
    } else {
        ce = cudaFuncSetAttribute(ssf_sparse_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (ce == cudaSuccess) ssf_sparse_kernel<false><<<grid, 32 * chains, smem, ctx->stream>>>(p);
    }
    if (ce == cudaSuccess) ce = cudaGetLastError();
    if (ce != cudaSuccess) return fail(ctx, ISB_ERR_CUDA, "ssf_sparse_kernel launch failed: %s", cudaGetErrorString(ce));
    e->last_launches += 1;
    return ISB_OK;
}

}  // namespace isb
