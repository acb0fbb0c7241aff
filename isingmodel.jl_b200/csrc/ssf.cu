// ssf.cu — host launcher of the single-spin-flip sweep kernel (K1) plus the small dense kernels
// around it (K2): full local field J s + h (src/SpinSystems.jl:75-78), energy (:68-71),
// magnetisation, and the Philox dump kernels used by the parity tests.
#include <math.h>
#include <stdlib.h>

#include <algorithm>
#include <vector>

#include "handles.hpp"
#include "ssf_kernel.cuh"

namespace isb {

int ssf_cold_chains(const isb_ctx *ctx, int npad, bool fixed);                // ssf_cold.cu
cudaError_t launch_ssf_cold(const SsfParams &p, int chains, bool fixed, cudaStream_t st);
cudaError_t launch_ssf_dd(const SsfParams &p, int npl, bool list, bool tma, int grid, int threads, size_t smem,
                          cudaStream_t st);
cudaError_t launch_ssf_ff(const SsfParams &p, int npl, bool list, bool tma, int grid, int threads, size_t smem,
                          cudaStream_t st);
cudaError_t launch_ssf_ii(const SsfParams &p, int npl, int grid, int threads, cudaStream_t st);

size_t ssf_field_elem_size(const isb_model *m) { return m->prec == ISB_PREC_F32 ? sizeof(float) : sizeof(double); }

// ------------------------------------------------------------------ K2: dense field / energy kernels
// g_i = sum_j J[i][j] s_j summed sequentially over ascending j in double — the same order as the
// reference's generic row dot, so the initial fields are bit-identical to the oracle's for any J.
// J is symmetric (enforced at model creation), so thread i reads J[j][i]: coalesced across i.
template <bool ROUNDJ>
__device__ __forceinline__ double row_dot(const double *__restrict__ J, int npad, int n, const int8_t *s_sh, int i) {
    double acc = 0.0;
    for (int j = 0; j < n; ++j) {
        double v = J[(int64_t)j * npad + i];
        if (ROUNDJ) v = (double)(float)v;
        acc += v * (double)s_sh[j];
    }
    return acc;
}

template <typename HT, bool ROUNDJ>
__global__ void field_init_kernel(const double *__restrict__ J, const double *__restrict__ h, const int8_t *spins,
                                  int64_t lds, HT *fields, int n, int npad, double hsign) {
    extern __shared__ int8_t s_sh[];
    const int r = blockIdx.y;
    for (int j = threadIdx.x; j < npad; j += blockDim.x) s_sh[j] = spins[(int64_t)r * lds + j];
    __syncthreads();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npad) return;
    double v = 0.0;
    if (i < n) {
        const double g = row_dot<ROUNDJ>(J, npad, n, s_sh, i);
        v = hsign > 0 ? g + h[i] : g - h[i];
    }
    fields[(int64_t)r * npad + i] = (HT)v;
}

// Fixed-point fields F_i = sum_j Jint[i][j] s_j (no h: the decision adds it, csrc/ssf_kernel.cuh fixed_thresholds).
// Integer sums do not depend on the order, so a CTA reads its columns of J once for FI_RB replicas: thread p owns position
// p of the permuted rows (coalesced) and, J being symmetric, sums column p of Jint = row site(p).  sum over the spins
// that are up, doubled, minus the plain sum: one predicated add per coupling and replica.
constexpr int FI_RB = 16;
__global__ void __launch_bounds__(256) fixed_field_init_kernel(const int32_t *__restrict__ Jfix, const int8_t *spins,
                                                               int64_t lds, int32_t *fields, int npad, int R, int vec) {
    extern __shared__ uint32_t up_bits[];   // [FI_RB][npad / 32]: bit j % 32 of word j / 32 = spin j of the replica is up
    const int nw32 = npad >> 5, r0 = blockIdx.y * FI_RB;
    for (int idx = threadIdx.x; idx < FI_RB * nw32; idx += blockDim.x) {
        const int rr = r0 + idx / nw32, w = idx % nw32;
        uint32_t b = 0;
        if (rr < R)
            for (int l = 0; l < 32; ++l) b |= (spins[(int64_t)rr * lds + w * 32 + l] > 0 ? 1u : 0u) << l;
        up_bits[idx] = b;
    }
    __syncthreads();
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    int32_t up[FI_RB], all = 0;
#pragma unroll
    for (int r = 0; r < FI_RB; ++r) up[r] = 0;
    for (int w = 0; w < nw32; ++w) {
        uint32_t bw[FI_RB];
#pragma unroll
        for (int r = 0; r < FI_RB; ++r) bw[r] = up_bits[r * nw32 + w];
#pragma unroll 4
        for (int l = 0; l < 32; ++l) {
            const int32_t v = __ldg(&Jfix[(int64_t)(w * 32 + l) * npad + p]);
            all += v;
#pragma unroll
            for (int r = 0; r < FI_RB; ++r) up[r] += ((bw[r] >> l) & 1u) ? v : 0;
        }
    }
    const int site = ssf_perm_site(p, vec);
#pragma unroll
    for (int r = 0; r < FI_RB; ++r)
        if (r0 + r < R) fields[(int64_t)(r0 + r) * npad + site] = 2 * up[r] - all;   // (wrap-around: exact in range)
}

__global__ void dense_field_kernel(const double *__restrict__ J, const double *__restrict__ h, const int8_t *spins,
                                   int64_t lds, double *out, int64_t ldo, int n, int npad) {
    extern __shared__ int8_t s_sh[];
    const int r = blockIdx.y;
    for (int j = threadIdx.x; j < npad; j += blockDim.x) s_sh[j] = spins[(int64_t)r * lds + j];
    __syncthreads();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    out[(int64_t)r * ldo + i] = row_dot<false>(J, npad, n, s_sh, i) + h[i];
}

// E_r = -1/2 sum_i s_i g_i - sum_i h_i s_i ; one CTA per replica, tree reduction of the outer sums.
__global__ void dense_energy_kernel(const double *__restrict__ J, const double *__restrict__ h, const int8_t *spins,
                                    int64_t lds, double *E, int n, int npad) {
    extern __shared__ int8_t s_sh[];
    __shared__ double red_q[32], red_l[32];
    const int r = blockIdx.x;
    for (int j = threadIdx.x; j < npad; j += blockDim.x) s_sh[j] = spins[(int64_t)r * lds + j];
    __syncthreads();
    double q = 0.0, l = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const double si = (double)s_sh[i];
        q += si * row_dot<false>(J, npad, n, s_sh, i);
        l += h[i] * si;
    }
    q = warp_sum(q);
    l = warp_sum(l);
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) {
        red_q[w] = q;
        red_l[w] = l;
    }
    __syncthreads();
    if (w == 0) {
        const int nwarp = blockDim.x >> 5;
        q = lane < nwarp ? red_q[lane] : 0.0;
        l = lane < nwarp ? red_l[lane] : 0.0;
        q = warp_sum(q);
        l = warp_sum(l);
        if (lane == 0) E[r] = -0.5 * q - l;
    }
}

__global__ void magnetization_kernel(const int8_t *spins, int64_t lds, int n, int R, double *M) {
    const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (r >= R) return;
    int m = 0;
    for (int i = lane; i < n; i += 32) m += spins[(int64_t)r * lds + i];
    m = warp_sum_int(m);
    if (lane == 0) M[r] = (double)m;
}

// ------------------------------------------------------------------ Philox dump kernels (parity tests)
__global__ void philox_fluct_kernel(int rule, uint64_t seed, uint64_t step_offset, int r0, int nr, int64_t nsteps,
                                    double *out) {
    const int64_t total = (int64_t)nr * nsteps;
    for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total;
         idx += (int64_t)gridDim.x * blockDim.x) {
        const int rr = (int)(idx / nsteps);
        const int64_t k = idx % nsteps;
        out[idx] = ssf_fluct_from_word(
            rule, philox_step_word(seed, DOM_SSF_FLUCT, (uint32_t)(r0 + rr), step_offset + (uint64_t)k));
    }
}
__global__ void philox_nodes_kernel(int n, uint64_t seed, uint64_t step_offset, int64_t nsteps, int32_t *out) {
    for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < nsteps;
         k += (int64_t)gridDim.x * blockDim.x)
        out[k] = node_from_word(philox_step_word(seed, DOM_SSF_NODES, 0u, step_offset + (uint64_t)k), n);
}
__global__ void philox_raw_kernel(const uint32_t *ctr, uint32_t k0, uint32_t k1, int nblocks, uint32_t *out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nblocks) return;
    const Philox4 p = philox4x32_10(ctr[4 * i], ctr[4 * i + 1], ctr[4 * i + 2], ctr[4 * i + 3], k0, k1);
    out[4 * i] = p.x;
    out[4 * i + 1] = p.y;
    out[4 * i + 2] = p.z;
    out[4 * i + 3] = p.w;
}

static int grid_for(int64_t total, int threads) {
    int64_t g = (total + threads - 1) / threads;
    return (int)std::max<int64_t>(1, std::min<int64_t>(g, 148 * 16));
}

int philox_fluct_device(isb_ctx *ctx, int rule, uint64_t seed, uint64_t step_offset, int r0, int nr,
                        int64_t nsteps, double *d_out) {
    if ((int64_t)nr * nsteps == 0) return ISB_OK;
    philox_fluct_kernel<<<grid_for((int64_t)nr * nsteps, 256), 256, 0, ctx->stream>>>(rule, seed, step_offset, r0, nr,
                                                                                      nsteps, d_out);
    ISB_CUDA(ctx, cudaGetLastError());
    return ISB_OK;
}
int philox_nodes_device(isb_ctx *ctx, int n, uint64_t seed, uint64_t step_offset, int64_t nsteps, int32_t *d_out) {
    if (nsteps == 0) return ISB_OK;
    philox_nodes_kernel<<<grid_for(nsteps, 256), 256, 0, ctx->stream>>>(n, seed, step_offset, nsteps, d_out);
    ISB_CUDA(ctx, cudaGetLastError());
    return ISB_OK;
}
int philox_raw_device(isb_ctx *ctx, const uint32_t *d_ctr, uint32_t k0, uint32_t k1, int nblocks, uint32_t *d_out) {
    if (nblocks == 0) return ISB_OK;
    philox_raw_kernel<<<(nblocks + 127) / 128, 128, 0, ctx->stream>>>(d_ctr, k0, k1, nblocks, d_out);
    ISB_CUDA(ctx, cudaGetLastError());
    return ISB_OK;
}

int dense_energy_device(isb_ens *e, double *d_E) {
    isb_model *m = e->model;
    dense_energy_kernel<<<e->R, 256, m->npad, m->ctx->stream>>>(m->J64, m->h64, e->spins, e->lds, d_E, m->n, m->npad);
    ISB_CUDA(m->ctx, cudaGetLastError());
    return ISB_OK;
}
int dense_field_device(isb_ens *e, double *d_F, int64_t ld) {
    isb_model *m = e->model;
    dim3 grid((m->n + 255) / 256, e->R);
    dense_field_kernel<<<grid, 256, m->npad, m->ctx->stream>>>(m->J64, m->h64, e->spins, e->lds, d_F, ld, m->n,
                                                               m->npad);
    ISB_CUDA(m->ctx, cudaGetLastError());
    return ISB_OK;
}
int magnetization_device(isb_ens *e, double *d_M) {
    isb_model *m = e->model;
    const int n = (m->kind == ISB_KIND_DENSE || m->kind == ISB_KIND_SPARSE) ? m->n : m->nv;
    magnetization_kernel<<<(e->R + 7) / 8, 256, 0, m->ctx->stream>>>(e->spins, e->lds, n, e->R, d_M);
    ISB_CUDA(m->ctx, cudaGetLastError());
    return ISB_OK;
}

// Configuration histogram (demo.jl:159-168): index = sum_i ((1 - s_i)/2) << (n-1-i).  Small state spaces are
// counted in shared memory first (every replica hits the same few bins), large ones go straight to global atomics.
template <bool SMEM>
__global__ void config_histogram_kernel(const int8_t *__restrict__ S, int64_t count, int n,
                                        unsigned long long *__restrict__ hist) {
    extern __shared__ unsigned int bins[];
    const unsigned nb = 1u << n;
    if (SMEM) {
        for (unsigned b = threadIdx.x; b < nb; b += blockDim.x) bins[b] = 0u;
        __syncthreads();
    }
    for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < count; c += (int64_t)gridDim.x * blockDim.x) {
        const int8_t *s = S + c * n;
        unsigned idx = 0;
        for (int i = 0; i < n; ++i) idx = (idx << 1) | (s[i] < 0 ? 1u : 0u);
        if (SMEM) atomicAdd(&bins[idx], 1u);
        else atomicAdd(&hist[idx], 1ull);
    }
    if (SMEM) {
        __syncthreads();
        for (unsigned b = threadIdx.x; b < nb; b += blockDim.x)
            if (bins[b]) atomicAdd(&hist[b], (unsigned long long)bins[b]);
    }
}
int config_histogram_device(isb_ctx *ctx, const int8_t *d_S, int64_t count, int n, unsigned long long *d_hist) {
    if (count == 0) return ISB_OK;
    const int blocks = (int)std::min<int64_t>((count + 255) / 256, 148 * 8);
    if (n <= 12)
        config_histogram_kernel<true><<<blocks, 256, sizeof(unsigned int) << n, ctx->stream>>>(d_S, count, n, d_hist);
    else
        config_histogram_kernel<false><<<blocks, 256, 0, ctx->stream>>>(d_S, count, n, d_hist);
    ISB_CUDA(ctx, cudaGetLastError());
    return ISB_OK;
}

// (Re)compute the cached local fields for the given h sign (+1: J s + h, -1: J s - h).
int ssf_ensure_fields(isb_ens *e, int sign) {
    isb_model *m = e->model;
    if (e->steps_since_refresh >= (int64_t)ISB_FIELD_REFRESH_SWEEPS * m->n) e->fields_rule_sign = 0;  // bound the drift
    if (e->fields_rule_sign == sign) return ISB_OK;
    e->steps_since_refresh = 0;
    dim3 grid((m->npad + 255) / 256, e->R);
    const double hs = (double)sign;
    if (m->prec == ISB_PREC_F32) {
        field_init_kernel<float, true><<<grid, 256, m->npad, m->ctx->stream>>>(
            m->J64, m->h64, e->spins, e->lds, (float *)e->fields, m->n, m->npad, hs);
    } else {
        field_init_kernel<double, false><<<grid, 256, m->npad, m->ctx->stream>>>(
            m->J64, m->h64, e->spins, e->lds, (double *)e->fields, m->n, m->npad, hs);
    }
    ISB_CUDA(m->ctx, cudaGetLastError());
    e->fields_rule_sign = sign;
    e->last_launches += 1;
    return ISB_OK;
}

// (Re)compute the cached fixed-point fields (they do not depend on h or the rule, and never drift).
static int ssf_ensure_fixed_fields(isb_ens *e) {
    isb_model *m = e->model;
    isb_ctx *ctx = m->ctx;
    if (!e->ifields) ISB_CUDA(ctx, cudaMalloc(&e->ifields, (size_t)e->R * m->npad * sizeof(int32_t)));
    if (e->ifields_ok) return ISB_OK;
    const int threads = std::min(m->npad, 256);
    dim3 grid(m->npad / threads, (e->R + FI_RB - 1) / FI_RB);
    fixed_field_init_kernel<<<grid, threads, FI_RB * (m->npad / 32) * sizeof(uint32_t), ctx->stream>>>(
        m->Jfix, e->spins, e->lds, e->ifields, m->npad, e->R, std::min(4, m->npl));
    ISB_CUDA(ctx, cudaGetLastError());
    e->ifields_ok = true;
    e->last_launches += 1;
    return ISB_OK;
}

// ------------------------------------------------------------------ K1 launch
static int ssf_run_device(isb_ens *e, int rule, int64_t nsteps, int order, const int32_t *d_nodes, int start,
                          int fluct_mode, const double *d_fluct, uint64_t seed, uint64_t step_offset,
                          const double *d_T, int64_t steps_per_T, int64_t trace_every, double *d_E, double *d_M, int8_t *d_S) {
    isb_model *m = e->model;
    isb_ctx *ctx = m->ctx;
    if (!m->fast_ok)
        return fail(ctx, ISB_ERR_UNSUPPORTED, "single-spin sweeps support N <= 1024 sites (N = %d)", m->n);
    if (nsteps <= 0) return ISB_OK;
    const bool list = order != ISB_ORDER_SEQUENTIAL;
    // The fixed-point kernels (int32 couplings and fields, exact fallback at the decision boundary: DESIGN §3) take every
    // untraced sequential run of a model that allows them; traces (energies compared at 1e-9) and the tie audit keep the
    // Float64 kernels.  ISB_SSF_FIXED=0 forces the Float64 path (A/B runs).
    bool fixed = m->fixed_ok && !list && trace_every == 0 && e->tie_eps == 0.0;
    if (const char *env_fx = getenv("ISB_SSF_FIXED")) fixed = fixed && atoi(env_fx) != 0;
    // a run on one path leaves the other path's cache stale
    int rc = fixed ? ssf_ensure_fixed_fields(e) : ssf_ensure_fields(e, rule == ISB_RULE_HOPFIELD ? -1 : +1);
    if (rc) return rc;
    if (fixed)
        e->fields_rule_sign = 0;
    else
        e->ifields_ok = false;

    const bool hd = m->prec != ISB_PREC_F32;
    const bool jf = m->j_is_f32;
    const int npl = m->npl;
    const int jsize = jf ? 4 : 8;
    const int rowb = m->npad * jsize;
    const int max_chains = fixed ? SSF_FIXED_CHAINS : ssf_max_chains(npl * (hd ? 2 : 1));

    int ctas, nw;
    if (e->R <= ctx->num_sms) {
        ctas = e->R;
        nw = 1;
    } else {
        const int waves = (e->R + ctx->num_sms * max_chains - 1) / (ctx->num_sms * max_chains);
        ctas = ctx->num_sms * waves;
        nw = (e->R + ctas - 1) / ctas;
        ctas = (e->R + nw - 1) / nw;
    }
    const int NG = std::min(8, (int)((ctx->smem_optin - 2048) / ((size_t)SSF_G * rowb)));
    // the fixed-point path has no streaming kernel: with 4 KiB rows the plain kernel (rows from L1 / L2) was faster than a
    // TMA ring at every acceptance of the C2 anneal (38 % down to 0.1 %; profiles/ssf_fixed_ab_b200.json)
    const bool tma = NG >= 2 && !fixed;
    // ring | full and empty barrier per slot, epoch and go barrier | epoch flips and mode
    const size_t smem = tma ? (size_t)NG * SSF_G * rowb + (size_t)(2 * NG + 2) * sizeof(uint64_t) + 16 : 0;

    SsfParams p{};
    p.J = fixed ? (const void *)m->Jfix : m->Jperm;
    p.ldj = m->npad;
    p.hext = m->h64;
    p.spins = e->spins;
    p.lds = e->lds;
    p.fields = fixed ? (void *)e->ifields : e->fields;
    p.n = m->n;
    p.npad = m->npad;
    p.R = e->R;
    p.rule = rule;
    p.ecoef = rule == ISB_RULE_HOPFIELD ? 1.5 : 0.5;
    p.nsteps = nsteps;
    p.start = start;
    p.nodes = d_nodes;
    p.fluct_mode = fluct_mode;
    p.fluct = d_fluct;
    p.seed = seed;
    p.step_offset = step_offset;
    p.Tsched = d_T;
    p.tscale = e->d_tscale;
    p.steps_per_T = steps_per_T;
    p.trace_every = trace_every;
    p.out_E = d_E;
    p.out_M = d_M;
    p.out_S = d_S;
    p.ldS = m->n;
    p.flips = e->d_flips;
    p.near_ties = e->d_counters;
    p.fallbacks = e->d_counters + 1;
    p.fix_q = m->fix_q;
    p.fix_invq = 1.0 / m->fix_q;   // (a power of two: exact)
    p.fix_margin = m->fix_margin;
    p.tie_eps = e->tie_eps;
    p.nw = nw;
    p.NG = NG;
    p.keys = philox_keys(seed);
    p.guard = m->guard;
    p.J64 = m->J64;
    p.ld64 = m->npad;
    p.hsign = rule == ISB_RULE_HOPFIELD ? -1.0 : 1.0;
    p.od_ratio = 0.8f;

    p.fluct_pitch = nsteps;
    const int threads = 32 * (nw + (fixed ? 0 : 1));   // (+ the producer warp of the ring kernels)
    // one launch over the steps [t0, t0 + len) of the run: every per-step input is offset on the host, the kernel sees a
    // run of `len` steps (t0 is a multiple of steps_per_T and of trace_every, see below)
    // mode 2: streaming kernel (TMA ring); 1: plain kernel (rows on demand, fields in registers); 0: cold kernel (fields in
    // shared memory, 28 chains per SM: ssf_cold.cu)
    const int cold_chains = fixed ? ssf_cold_chains(ctx, m->npad, true)
                            : (hd && !jf && !list && trace_every == 0 && p.guard == 0.0 && p.tie_eps == 0.0)
                                ? ssf_cold_chains(ctx, m->npad, false) : 0;
    auto launch = [&](int64_t t0, int64_t len, int mode) -> cudaError_t {
        const bool use_tma = mode == 2;
        SsfParams q = p;
        q.nsteps = len;
        q.step_offset = step_offset + (uint64_t)t0;
        if (list) {
            q.nodes = d_nodes + t0;
        } else {
            q.start = (int)(((int64_t)start + t0) % m->n);
        }
        if (d_fluct) q.fluct = d_fluct + t0;                 // (shared: step t0; per replica: [r][t0], pitch = whole run)
        q.Tsched = d_T + t0 / steps_per_T;
        if (trace_every > 0) {
            const int64_t i0 = t0 / trace_every;
            if (d_E) q.out_E = d_E + i0 * e->R;
            if (d_M) q.out_M = d_M + i0 * e->R;
            if (d_S) q.out_S = d_S + i0 * e->R * (int64_t)m->n;
        }
        if (mode == 0) return launch_ssf_cold(q, cold_chains, fixed, ctx->stream);
        const size_t sm = use_tma ? smem : 0;
        if (fixed) return launch_ssf_ii(q, npl, ctas, threads, ctx->stream);
        return hd ? launch_ssf_dd(q, npl, list, use_tma, ctas, threads, sm, ctx->stream)
                  : launch_ssf_ff(q, npl, list, use_tma, ctas, threads, sm, ctx->stream);
    };
    // Adaptive delivery across launches.  The streaming kernel (TMA ring, adaptive epochs) wins while more than about one
    // flip in five is accepted; below that the plain kernel — every chain reads the rows of its own flips from L2, no
    // producer warp, no epoch synchronisation between the chains of a CTA — is up to 1.7x faster per sweep (C2 schedule,
    // profiles/r2aq_c2_delivery_profile.txt).  Sequential sweeps longer than two segments are therefore run segment by
    // segment, each in the mode the previous segment's acceptance calls for; the fields stay cached on the device between
    // launches and the trajectory does not depend on the segmentation (noise, schedule and traces are indexed by the
    // step of the run).  ISB_SSF_SEGMENT=0 keeps one launch.
    int64_t unit = steps_per_T;
    if (trace_every > 0) {   // least common multiple of the schedule period and the trace period
        int64_t a = unit, b = trace_every;
        while (b) {
            const int64_t c = a % b;
            a = b;
            b = c;
        }
        unit = unit / a * trace_every;
    }
    int64_t seg = std::max<int64_t>((int64_t)50 * m->n, (int64_t)1 << 16);
    double min_work = 1e5;   // replicas x sites below which a launch is too short to be worth splitting
    if (const char *env_sm = getenv("ISB_SSF_SEG_MIN")) {   // tests: segment length in steps, any problem size
        seg = std::max<int64_t>(1, atoll(env_sm));
        min_work = 0.0;
    }
    seg = (seg + unit - 1) / unit * unit;
    bool segment = (tma || fixed) && !list && unit > 0 && nsteps > 2 * seg && (double)e->R * m->n >= min_work;
    if (const char *env_sg = getenv("ISB_SSF_SEGMENT")) segment = segment && atoi(env_sg) != 0;
    double thr = fixed ? 2.0 : 0.2;   // accepted flips per attempt above which the streaming kernel is the faster one
    if (const char *env_th = getenv("ISB_SSF_SEG_THR")) thr = atof(env_th);
    cudaError_t ce = cudaSuccess;
    // ... below which the shared-memory-field kernel is the fastest (one wave of 28 chains per SM).  Fixed point: the cold
    // kernel overtakes the plain one between 2.8 % and 2.0 % acceptance (C2 profile, profiles/ssf_fixed_ab_b200.json)
    double thr_cold = 0.03;
    if (const char *env_tc = getenv("ISB_SSF_COLD_THR")) thr_cold = atof(env_tc);
    if (cold_chains < 16) thr_cold = -1.0;
    // ISB_SSF_MODE = 0 | 1 | 2: one launch of that kernel (A/B runs and tests).  A mode the run cannot take is an error, so
    // that a test which forces a kernel never passes on another one.
    int forced = -1;
    if (const char *env_md = getenv("ISB_SSF_MODE")) {
        forced = atoi(env_md);
        if (forced < 0 || forced > 2)
            return fail(ctx, ISB_ERR_ARG, "ISB_SSF_MODE=%s: expected 0 (cold), 1 (plain) or 2 (streaming)", env_md);
        if (forced == 0 && cold_chains < 1)
            return fail(ctx, ISB_ERR_ARG,
                        "ISB_SSF_MODE=0: no cold kernel for this run (it needs sequential order, no traces, no tie audit, and "
                        "either fixed point with Npad %% 128 == 0 or Float64 without the near-tie guard with Npad %% 64 == 0; "
                        "Npad = %d, %s)", m->npad, fixed ? "fixed point" : (hd ? "Float64" : "Float32"));
        if (forced == 2 && !tma)
            return fail(ctx, ISB_ERR_ARG, "ISB_SSF_MODE=2: no streaming kernel for this run (%s)",
                        fixed ? "the fixed-point path has none" : "the ring does not fit in shared memory");
    }
    if (forced >= 0) {
        ce = launch(0, nsteps, forced);
        e->last_launches += 1;
    } else if (!segment) {
        ce = launch(0, nsteps, tma ? 2 : 1);
        e->last_launches += 1;
    } else {
        std::vector<unsigned long long> fl((size_t)e->R), tot((size_t)e->R, 0ull);
        int mode = tma ? 2 : 1;
        int stable = 0;
        for (int64_t t0 = 0; t0 < nsteps && ce == cudaSuccess;) {
            const int64_t len = std::min(seg, nsteps - t0);
            ce = launch(t0, len, mode);
            e->last_launches += 1;
            if (ce != cudaSuccess) break;
            ce = cudaMemcpyAsync(fl.data(), e->d_flips, fl.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream);
            if (ce == cudaSuccess) ce = cudaStreamSynchronize(ctx->stream);
            if (ce != cudaSuccess) break;
            double sum = 0.0;
            for (size_t r = 0; r < fl.size(); ++r) {
                tot[r] += fl[r];
                sum += (double)fl[r];
            }
            // (the decision lags one segment behind: in an anneal the acceptance of the next segment is lower still)
            const double acc = sum / ((double)len * e->R);
            const int next = acc > thr ? 2 : (acc > thr_cold ? 1 : 0);
            stable = next == mode ? stable + 1 : 0;
            mode = next;
            // a settled cold regime: fewer, longer launches.  Hot segments stay short — an anneal leaves them, and a long
            // streamed segment that has gone cold costs more than the extra launches
            if (mode == 0 && stable >= 2) seg = std::min<int64_t>(seg * 2, (int64_t)1 << 40);
            t0 += len;
        }
        if (ce == cudaSuccess)   // the flip counts of the whole run, where the caller reads them
            ce = cudaMemcpyAsync(e->d_flips, tot.data(), tot.size() * sizeof(unsigned long long), cudaMemcpyHostToDevice, ctx->stream);
        if (ce == cudaSuccess) ce = cudaStreamSynchronize(ctx->stream);
    }
    if (ce != cudaSuccess)
        return fail(ctx, ISB_ERR_CUDA, "ssf_kernel launch failed: %s (grid %d x %d threads, %zu B smem)",
                    cudaGetErrorString(ce), ctas, threads, smem);
    e->steps_since_refresh += nsteps;
    return ISB_OK;
}

int ssf_sweep_device(isb_ens *e, int rule, int64_t nsteps, int order, int32_t *d_nodes, int start, int fluct_mode,
                     const double *d_fluct, uint64_t seed, uint64_t step_offset, const double *d_T, int64_t steps_per_T,
                     int64_t trace_every, double *d_E, double *d_M, int8_t *d_S) {
    isb_model *m = e->model;
    if (order == ISB_ORDER_RANDOM) {
        if (int rc = philox_nodes_device(m->ctx, m->n, seed, step_offset, nsteps, d_nodes)) return rc;
        e->last_launches += 1;
    }
    if (m->kind == ISB_KIND_SPARSE || !m->fast_ok)
        return ssf_sparse_run_device(e, rule, nsteps, order, d_nodes, start, fluct_mode, d_fluct, seed, step_offset, d_T,
                                     steps_per_T, trace_every, d_E, d_M, d_S);
    return ssf_run_device(e, rule, nsteps, order, d_nodes, start, fluct_mode, d_fluct, seed, step_offset, d_T, steps_per_T,
                          trace_every, d_E, d_M, d_S);
}

}  // namespace isb
