// api.cu — the extern "C" surface of libising_b200.so (include/ising_b200.h): contexts, models,
// ensembles, host<->device staging and the run entry points.  No torch types, no CPU compute path:
// every entry point that produces spins, fields or energies launches a CUDA kernel.
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "handles.hpp"

// Error texts are per THREAD (and remember which context they belong to): two threads that share a context, or use
// two contexts, each read the message of their own last failed call.
static thread_local std::string g_create_err = "";
static thread_local std::string g_ctx_err = "";
static thread_local const isb_ctx *g_ctx_err_owner = nullptr;

namespace isb {

int fail(isb_ctx *ctx, int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (ctx) {
        g_ctx_err = buf;
        g_ctx_err_owner = ctx;
    } else {
        g_create_err = buf;
    }
    return code;
}

// absrowsum[i] = sum_j |J_ij| + |h_i|; vals = every coupling (any order), h = the fields
double ssf_guard_from(const double *absrowsum, const double *vals, size_t nvals, const double *h, int n) {
    // exact arithmetic: every value is an integer multiple of 2^-20 and the row sums stay below 2^30 -> every partial sum
    // (and its doubling) is exactly representable, the incremental field equals the fresh row dot bit for bit
    bool exact = true;
    double big = 0.0;
    auto dyadic = [](double v) {
        const double s = v * 1048576.0;
        return std::fabs(s) < 4503599627370496.0 && s == std::nearbyint(s);
    };
    for (size_t k = 0; k < nvals && exact; ++k) exact = dyadic(vals[k]);
    for (int i = 0; i < n; ++i) {
        if (exact && h) exact = dyadic(h[i]);
        big = std::max(big, absrowsum[i]);
    }
    if (exact && big < 1073741824.0) return 0.0;
    // couplings drawn from a continuum (more than 64 distinct magnitudes): an exact tie or cancellation of the reference
    // has probability zero, and so has a decision within an ulp of one; no guard (the near-tie audit still counts them)
    std::vector<double> mags;
    for (size_t k = 0; k < nvals; ++k) {
        const double a = std::fabs(vals[k]);
        if (a == 0.0) continue;
        if (std::find(mags.begin(), mags.end(), a) == mags.end()) {
            mags.push_back(a);
            if (mags.size() > 64) return 0.0;
        }
    }
    return std::ldexp(big > 0.0 ? big : 1.0, -30);
}

int dev_reserve(isb_ctx *ctx, int slot, size_t bytes, void **out) {
    isb_devbuf &b = ctx->scratch[slot];
    if (bytes == 0) bytes = 16;
    if (b.cap < bytes) {
        if (b.p) {
            ISB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
            ISB_CUDA(ctx, cudaFree(b.p));
            b.p = nullptr;
            b.cap = 0;
        }
        const size_t cap = std::max(bytes, (size_t)4096);
        ISB_CUDA(ctx, cudaMalloc(&b.p, cap));
        b.cap = cap;
    }
    *out = b.p;
    return ISB_OK;
}

}  // namespace isb

using isb::fail;

#define ISB_TRY(expr)            \
    do {                         \
        int _rc = (expr);        \
        if (_rc != ISB_OK) return _rc; \
    } while (0)

static bool all_finite(const double *p, size_t n) {
    for (size_t i = 0; i < n; ++i)
        if (!std::isfinite(p[i])) return false;
    return true;
}

static int h2d(isb_ctx *ctx, void *dst, const void *src, size_t bytes, int64_t *acc) {
    if (bytes == 0) return ISB_OK;
    ISB_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    if (acc) *acc += (int64_t)bytes;
    return ISB_OK;
}
static int d2h(isb_ctx *ctx, void *dst, const void *src, size_t bytes, int64_t *acc) {
    if (bytes == 0) return ISB_OK;
    ISB_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    if (acc) *acc += (int64_t)bytes;
    return ISB_OK;
}

extern "C" {

// ------------------------------------------------------------------ context
int isb_version(void) { return ISB_VERSION; }

int isb_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int isb_create(int device, isb_ctx **out) {
    if (!out) return fail(nullptr, ISB_ERR_ARG, "isb_create: out is NULL");
    *out = nullptr;
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(nullptr, ISB_ERR_CUDA,
                    "isb_create: no CUDA device (%s); libising_b200 has no CPU fallback",
                    ce == cudaSuccess ? "device count is 0" : cudaGetErrorString(ce));
    }
    if (device < 0 || device >= ndev)
        return fail(nullptr, ISB_ERR_ARG, "isb_create: device %d out of range [0, %d)", device, ndev);
    ISB_CUDA(nullptr, cudaSetDevice(device));
    int major = 0, sms = 0, optin = 0;
    ISB_CUDA(nullptr, cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
    ISB_CUDA(nullptr, cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    ISB_CUDA(nullptr, cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
    if (major != 10)
        return fail(nullptr, ISB_ERR_CUDA, "isb_create: device %d is sm_%d0; this library is built for sm_100a only",
                    device, major);
    isb_ctx *ctx = new isb_ctx();
    ctx->device = device;
    ctx->num_sms = sms;
    ctx->smem_optin = (size_t)optin;
    ISB_CUDA(nullptr, cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    ctx->own_stream = true;
    ISB_CUDA(nullptr, cudaEventCreate(&ctx->ev0));
    ISB_CUDA(nullptr, cudaEventCreate(&ctx->ev1));
    *out = ctx;
    return ISB_OK;
}

// Handles are reference counted so that destruction order does not matter to the caller (a garbage
// collector may release a model before the ensembles that use it).
static void ctx_release(isb_ctx *ctx) {
    if (!ctx || ctx->refs.fetch_sub(1) != 1) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    for (auto &b : ctx->scratch)
        if (b.p) cudaFree(b.p);
    if (ctx->ev0) cudaEventDestroy(ctx->ev0);
    if (ctx->ev1) cudaEventDestroy(ctx->ev1);
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

void isb_destroy(isb_ctx *ctx) { ctx_release(ctx); }

const char *isb_last_error(const isb_ctx *ctx) {
    if (!ctx) return g_create_err.c_str();
    return g_ctx_err_owner == ctx ? g_ctx_err.c_str() : "";
}

int isb_set_stream(isb_ctx *ctx, void *cuda_stream) {
    if (!ctx) return ISB_ERR_ARG;
    ISB_LOCK(ctx);
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    ctx->stream = (cudaStream_t)cuda_stream;
    ctx->own_stream = false;
    return ISB_OK;
}

int isb_synchronize(isb_ctx *ctx) {
    if (!ctx) return ISB_ERR_ARG;
    ISB_LOCK(ctx);
    ISB_CUDA(ctx, cudaSetDevice(ctx->device));
    ISB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return ISB_OK;
}

// ------------------------------------------------------------------ models
static int next_pow2(int v) {
    int p = 1;
    while (p < v) p <<= 1;
    return p;
}

// Fixed-point couplings for the sweep kernels (DESIGN §3).  q = 2^-k with the largest k (|k| <= 1000) such that every row
// sum of |Jint| = |round(J / q)| stays below 2^30, so that the cached integer fields F = Jint s and every threshold of the
// kernels fit an int32.  M bounds, in units of q, how far the reference's own Float64 row dot can lie from F q:
//   |J s - q Jint s| <= e_i = sum_j |J_ij - q Jint_ij|   (each term exact, the sum rounded up by a factor 1 + 2^-40),
//   |dot_ref - J s|  <= (n - 1) 2^-53 sum_j |J_ij| < 2^-40 sum_j |J_ij|   (sequential sum of n <= 1024 exact products),
// M = ceil(max_i (e_i + 2^-40 sum_j |J_ij|) / q) + 1, and M = 0 when every coupling is a multiple of q (then every partial
// sum of the reference is an exact multiple of q below 2^30 q: its dot IS F q).  The model keeps the Float64 kernels when
// M > 2^-20 sum_j |Jint_ij| for some row with couplings (a fallback band wider than 2^-20 of that row's field scale:
// rows far weaker than the strongest one would fall back often) or when some |h_i| / q >= 2^50 (the reference's
// h_i + dot rounds at a step above q).  Jq: the permuted int32 rows (VEC = 4), like Jperm.
static bool fixed_point_couplings(const std::vector<double> &Jn, const std::vector<double> &hn, int n, int npad,
                                  std::vector<int32_t> *Jq, double *q_out, int *M_out) {
    double smax = 0.0, hmax = 0.0;
    for (int i = 0; i < n; ++i) {
        double s = 0.0;
        for (int j = 0; j < n; ++j) s += std::fabs(Jn[(size_t)i * npad + j]);
        smax = std::max(smax, s);
        hmax = std::max(hmax, std::fabs(hn[i]));
    }
    int k = smax > 0.0 ? (int)std::floor(std::log2(1073741824.0 / smax)) : 0;
    k = std::max(-1000, std::min(1000, k));
    std::vector<int64_t> Ji((size_t)n * n);
    for (;; --k) {
        if (k < -1000) return false;
        int64_t worst = 0;
        for (int i = 0; i < n; ++i) {
            int64_t s = 0;
            for (int j = 0; j < n; ++j) {
                const double v = std::nearbyint(std::ldexp(Jn[(size_t)i * npad + j], k));
                Ji[(size_t)i * n + j] = std::fabs(v) < 4e18 ? (int64_t)v : (int64_t)1 << 62;
                s += std::llabs(Ji[(size_t)i * n + j]);
                if (s >= ((int64_t)1 << 30)) break;
            }
            worst = std::max(worst, s);
        }
        if (worst < ((int64_t)1 << 30)) break;
    }
    const double q = std::ldexp(1.0, -k);
    double emax = 0.0;
    int64_t smin = (int64_t)1 << 30;   // smallest nonzero row sum of |Jint|
    bool exact = true;
    for (int i = 0; i < n; ++i) {
        double e = 0.0, s = 0.0;
        int64_t si = 0;
        for (int j = 0; j < n; ++j) {
            si += std::llabs(Ji[(size_t)i * n + j]);
            const double v = Jn[(size_t)i * npad + j];
            const double d = std::fabs(v - std::ldexp((double)Ji[(size_t)i * n + j], -k));  // exact (Sterbenz, or Jint = 0)
            exact = exact && d == 0.0;
            e += d;
            s += std::fabs(v);
        }
        emax = std::max(emax, e * (1.0 + 0x1p-40) + s * 0x1p-40);
        if (si > 0) smin = std::min(smin, si);
    }
    const double Md = exact ? 0.0 : std::ceil(emax / q) + 1.0;
    if (Md * 0x1p20 > (double)smin || hmax / q >= 0x1p50) return false;
    const int vec = std::min(4, npad / 32);
    Jq->assign((size_t)npad * npad, 0);
    for (int i = 0; i < n; ++i)
        for (int s = 0; s < n; ++s) (*Jq)[(size_t)i * npad + isb::ssf_perm_pos(s, vec)] = (int32_t)Ji[(size_t)i * n + s];
    *q_out = q;
    *M_out = (int)Md;
    return true;
}

int isb_model_dense(isb_ctx *ctx, int n, const double *J, int64_t ld, const double *h, int prec, int *warn,
                    isb_model **out) {
    if (!ctx) return ISB_ERR_ARG;
    ISB_LOCK(ctx);
    if (!out || !J) return fail(ctx, ISB_ERR_ARG, "isb_model_dense: NULL argument");
    *out = nullptr;
    if (warn) *warn = 0;
    if (n <= 0) return fail(ctx, ISB_ERR_SIZE, "isb_model_dense: n = %d must be positive", n);
    if (ld < n) return fail(ctx, ISB_ERR_SIZE, "isb_model_dense: leading dimension %lld < n = %d", (long long)ld, n);
    if (prec != ISB_PREC_F64 && prec != ISB_PREC_F32 && prec != ISB_PREC_AUTO)
        return fail(ctx, ISB_ERR_ARG, "isb_model_dense: prec must be ISB_PREC_F64, _F32 or _AUTO");
    ISB_CUDA(ctx, cudaSetDevice(ctx->device));

    const bool fast = n <= 1024;
    const int npl = fast ? next_pow2((n + 31) / 32) : 0;
    const int npad = fast ? 32 * npl : ((n + 31) / 32) * 32;
    std::vector<double> Jn((size_t)npad * npad, 0.0), hn((size_t)npad, 0.0);
    // symmetry / diagonal handling of src/SpinSystems.jl:31-38
    bool sym = true, diag = false;
    for (int j = 0; j < n && sym; ++j)
        for (int i = 0; i < j; ++i)
            if (J[i + (int64_t)j * ld] != J[j + (int64_t)i * ld]) {
                sym = false;
                break;
            }
    for (int j = 0; j < n; ++j) {
        for (int i = 0; i <= j; ++i) {
            const double up = J[i + (int64_t)j * ld];  // upper-triangle element; the lower one mirrors it: Symmetric(J, :U)
            if (!std::isfinite(up)) return fail(ctx, ISB_ERR_NONFINITE, "isb_model_dense: J[%d,%d] is not finite", i, j);
            if (i == j) {
                if (up != 0.0) diag = true;
                continue;
            }
            Jn[(size_t)i * npad + j] = up;
            Jn[(size_t)j * npad + i] = up;
        }
    }
    if (warn) *warn = (sym ? 0 : 1) | (diag ? 2 : 0);
    if (h) {
        if (!all_finite(h, (size_t)n)) return fail(ctx, ISB_ERR_NONFINITE, "isb_model_dense: h is not finite");
        for (int i = 0; i < n; ++i) hn[i] = h[i];
    }
    bool lossless_f32 = true;
    for (size_t k = 0; k < Jn.size() && lossless_f32; ++k) lossless_f32 = (double)(float)Jn[k] == Jn[k];

    isb_model *m = new isb_model();
    m->ctx = ctx;
    ctx->refs.fetch_add(1);
    m->kind = ISB_KIND_DENSE;
    m->prec = prec == ISB_PREC_AUTO ? ISB_PREC_F64 : prec;
    m->n = n;
    m->npad = npad;
    m->npl = npl;
    m->fast_ok = fast;
    // Float storage of J only together with float fields: measured on B200, float rows under Float64 fields are
    // SLOWER than double rows (227 vs 196 ms on the C2 schedule) — the 32 F2F conversions per row cost more than the
    // halved shared-memory traffic saves.  ISB_PREC_AUTO therefore means Float64 throughout for dense models.
    m->j_is_f32 = prec == ISB_PREC_F32;
    (void)lossless_f32;
    {
        std::vector<double> ars((size_t)n, 0.0);
        for (int i = 0; i < n; ++i) {
            double a = std::fabs(hn[i]);
            for (int j = 0; j < n; ++j) a += std::fabs(Jn[(size_t)i * npad + j]);
            ars[i] = a;
        }
        m->guard = prec == ISB_PREC_F32 ? 0.0 : isb::ssf_guard_from(ars.data(), Jn.data(), Jn.size(), hn.data(), n);
    }
    const size_t nn = (size_t)npad * npad;
    int rc = ISB_OK;
    do {
        if (cudaMalloc(&m->J64, nn * sizeof(double)) != cudaSuccess || cudaMalloc(&m->h64, npad * sizeof(double)) != cudaSuccess) {
            rc = fail(ctx, ISB_ERR_CUDA, "isb_model_dense: cudaMalloc failed: %s", cudaGetErrorString(cudaGetLastError()));
            break;
        }
        cudaMemcpyAsync(m->J64, Jn.data(), nn * sizeof(double), cudaMemcpyHostToDevice, ctx->stream);
        cudaMemcpyAsync(m->h64, hn.data(), npad * sizeof(double), cudaMemcpyHostToDevice, ctx->stream);
        if (fast) {
            // permuted copy for the sweep kernel (isb::ssf_perm_pos)
            const int jsz = m->j_is_f32 ? 4 : 8;
            const int vec = std::min(16 / jsz, npl);
            std::vector<unsigned char> Jp(nn * jsz);
            for (int i = 0; i < npad; ++i)
                for (int s = 0; s < npad; ++s) {
                    const size_t pos = (size_t)i * npad + isb::ssf_perm_pos(s, vec);
                    const double v = Jn[(size_t)i * npad + s];
                    if (m->j_is_f32)
                        reinterpret_cast<float *>(Jp.data())[pos] = (float)v;
                    else
                        reinterpret_cast<double *>(Jp.data())[pos] = v;
                }
            if (cudaMalloc(&m->Jperm, nn * jsz) != cudaSuccess) {
                rc = fail(ctx, ISB_ERR_CUDA, "isb_model_dense: cudaMalloc failed: %s", cudaGetErrorString(cudaGetLastError()));
                break;
            }
            cudaMemcpyAsync(m->Jperm, Jp.data(), nn * jsz, cudaMemcpyHostToDevice, ctx->stream);
            cudaStreamSynchronize(ctx->stream);
            std::vector<int32_t> Jq;
            if (m->prec == ISB_PREC_F64 && fixed_point_couplings(Jn, hn, n, npad, &Jq, &m->fix_q, &m->fix_margin)) {
                if (cudaMalloc(&m->Jfix, nn * sizeof(int32_t)) != cudaSuccess) {
                    rc = fail(ctx, ISB_ERR_CUDA, "isb_model_dense: cudaMalloc failed: %s", cudaGetErrorString(cudaGetLastError()));
                    break;
                }
                cudaMemcpyAsync(m->Jfix, Jq.data(), nn * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream);
                m->fixed_ok = true;
            }
        }
        cudaError_t ce = cudaStreamSynchronize(ctx->stream);
        if (ce != cudaSuccess) rc = fail(ctx, ISB_ERR_CUDA, "isb_model_dense: upload failed: %s", cudaGetErrorString(ce));
        if (!rc && !fast) {
            // N > 1024: the register-resident sweep kernel does not apply; sweeps run through the neighbour-list
            // kernel (sparse.cu) over the nonzero couplings, fields in shared memory
            std::vector<int64_t> colptr((size_t)n + 1, 0);
            std::vector<int32_t> rowval;
            std::vector<double> nzval;
            for (int j = 0; j < n; ++j) {
                for (int i = 0; i < n; ++i) {
                    const double v = Jn[(size_t)i * npad + j];
                    if (v != 0.0) {
                        rowval.push_back(i);
                        nzval.push_back(v);
                    }
                }
                colptr[j + 1] = (int64_t)rowval.size();
            }
            rc = isb::sparse_model_init(m, n, colptr.data(), rowval.data(), nzval.data(), nullptr);
            if (!rc) isb::sparse_model_set_guard(m, hn.data());
        }
    } while (0);
    if (rc) {
        isb_model_destroy(m);
        return rc;
    }
    *out = m;
    return ISB_OK;
}


int isb_model_sparse(isb_ctx *ctx, int n, const int64_t *colptr, const int32_t *rowval, const double *nzval,
                     const double *h, int *warn, isb_model **out) {
    if (!ctx) return ISB_ERR_ARG;
    ISB_LOCK(ctx);
    if (!out || !colptr) return fail(ctx, ISB_ERR_ARG, "isb_model_sparse: NULL argument");
    *out = nullptr;
    if (warn) *warn = 0;
    if (n <= 0) return fail(ctx, ISB_ERR_SIZE, "isb_model_sparse: n = %d must be positive", n);
    if (colptr[0] != 0) return fail(ctx, ISB_ERR_ARG, "isb_model_sparse: colptr[0] must be 0 (0-based CSC)");
    for (int j = 0; j < n; ++j)
        if (colptr[j + 1] < colptr[j]) return fail(ctx, ISB_ERR_ARG, "isb_model_sparse: colptr is not non-decreasing");
    if (colptr[n] > 0 && (!rowval || !nzval)) return fail(ctx, ISB_ERR_ARG, "isb_model_sparse: NULL argument");
    if (h && !all_finite(h, (size_t)n)) return fail(ctx, ISB_ERR_NONFINITE, "isb_model_sparse: h is not finite");
    ISB_CUDA(ctx, cudaSetDevice(ctx->device));
    isb_model *m = new isb_model();
    m->ctx = ctx;
    ctx->refs.fetch_add(1);
    m->kind = ISB_KIND_SPARSE;
    m->prec = ISB_PREC_F64;
    m->n = n;
    m->npad = (n + 31) / 32 * 32;
    std::vector<double> hn((size_t)m->npad, 0.0);
    if (h) std::copy(h, h + n, hn.begin());
    int rc = ISB_OK;
    if (cudaMalloc(&m->h64, m->npad * sizeof(double)) != cudaSuccess)
        rc = fail(ctx, ISB_ERR_CUDA, "isb_model_sparse: cudaMalloc failed");
    if (!rc) {
        cudaMemcpy(m->h64, hn.data(), m->npad * sizeof(double), cudaMemcpyHostToDevice);
        rc = isb::sparse_model_init(m, n, colptr, rowval, nzval, warn);
        if (!rc) isb::sparse_model_set_guard(m, hn.data());
    }
    if (rc) {
        isb_model_destroy(m);
        return rc;
    }
    *out = m;
    return ISB_OK;
}

int isb_model_bipartite(isb_ctx *ctx, int nv, int nh, const double *W, int64_t ld, const double *h, const double *b,
                        int prec, isb_model **out) {
    if (!ctx) return ISB_ERR_ARG;
    ISB_LOCK(ctx);
    if (!out || !W) return fail(ctx, ISB_ERR_ARG, "isb_model_bipartite: NULL argument");
    *out = nullptr;
    if (nv <= 0 || nh <= 0) return fail(ctx, ISB_ERR_SIZE, "isb_model_bipartite: nv = %d, nh = %d must be positive", nv, nh);
    if (ld < nv) return fail(ctx, ISB_ERR_SIZE, "isb_model_bipartite: leading dimension %lld < nv = %d", (long long)ld, nv);
    if (prec == ISB_PREC_AUTO) prec = ISB_PREC_F64;
    if (prec != ISB_PREC_F64 && prec != ISB_PREC_BF16X3 && prec != ISB_PREC_BF16X2 && prec != ISB_PREC_BF16X1 &&
        prec != ISB_PREC_FP16X2 && prec != ISB_PREC_FP16X1 && prec != ISB_PREC_I8X3 && prec != ISB_PREC_I8X2 && prec != ISB_PREC_I8X4)
        return fail(ctx, ISB_ERR_ARG, "isb_model_bipartite: prec must be ISB_PREC_F64, _BF16X3, _BF16X2, _BF16X1, _FP16X2, _FP16X1, _I8X3, _I8X2 or _I8X4");
    ISB_CUDA(ctx, cudaSetDevice(ctx->device));
    std::vector<double> Wr((size_t)nv * nh), Wt((size_t)nv * nh), hn((size_t)nv, 0.0), bn((size_t)nh, 0.0);
    for (int j = 0; j < nh; ++j)
        for (int i = 0; i < nv; ++i) {
            const double v = W[i + (int64_t)j * ld];
            if (!std::isfinite(v)) return fail(ctx, ISB_ERR_NONFINITE, "isb_model_bipartite: W[%d,%d] is not finite", i, j);
            Wr[(size_t)i * nh + j] = v;
            Wt[(size_t)j * nv + i] = v;
        }
    if (h) {
        if (!all_finite(h, nv)) return fail(ctx, ISB_ERR_NONFINITE, "isb_model_bipartite: h is not finite");
        std::copy(h, h + nv, hn.begin());
    }
    if (b) {
        if (!all_finite(b, nh)) return fail(ctx, ISB_ERR_NONFINITE, "isb_model_bipartite: b is not finite");
        std::copy(b, b + nh, bn.begin());
    }
    isb_model *m = new isb_model();
    m->ctx = ctx;
    ctx->refs.fetch_add(1);
    m->kind = ISB_KIND_BIPARTITE;
    m->prec = prec;
    m->nv = nv;
    m->nh = nh;
    int rc = ISB_OK;
    do {
        const size_t nn = (size_t)nv * nh * sizeof(double);
        if (cudaMalloc(&m->W64, nn) != cudaSuccess || cudaMalloc(&m->Wt64, nn) != cudaSuccess ||
            cudaMalloc(&m->hb64, nv * sizeof(double)) != cudaSuccess || cudaMalloc(&m->bb64, nh * sizeof(double)) != cudaSuccess) {
            rc = fail(ctx, ISB_ERR_CUDA, "isb_model_bipartite: cudaMalloc failed: %s", cudaGetErrorString(cudaGetLastError()));
            break;
        }
        cudaMemcpyAsync(m->W64, Wr.data(), nn, cudaMemcpyHostToDevice, ctx->stream);
        cudaMemcpyAsync(m->Wt64, Wt.data(), nn, cudaMemcpyHostToDevice, ctx->stream);
        cudaMemcpyAsync(m->hb64, hn.data(), nv * sizeof(double), cudaMemcpyHostToDevice, ctx->stream);
        cudaMemcpyAsync(m->bb64, bn.data(), nh * sizeof(double), cudaMemcpyHostToDevice, ctx->stream);
        cudaError_t ce = cudaStreamSynchronize(ctx->stream);
        if (ce != cudaSuccess) {
            rc = fail(ctx, ISB_ERR_CUDA, "isb_model_bipartite: upload failed: %s", cudaGetErrorString(ce));
            break;
        }
        if (prec != ISB_PREC_F64) rc = isb::bip_tc_model_init(m, Wr.data());
    } while (0);
    if (rc) {
        isb_model_destroy(m);
        return rc;
    }
    *out = m;
    return ISB_OK;
}

static void model_release(isb_model *m) {
    if (!m || m->refs.fetch_sub(1) != 1) return;
    isb_ctx *ctx = m->ctx;
    {
        ISB_LOCK(ctx);
        cudaSetDevice(ctx->device);
        cudaStreamSynchronize(ctx->stream);
        if (m->tc) isb::bip_tc_model_free(m);
        if (m->sp) isb::sparse_model_free(m);
        cudaFree(m->J64);
        cudaFree(m->Jperm);
        cudaFree(m->Jfix);
        cudaFree(m->h64);
        cudaFree(m->W64);
        cudaFree(m->Wt64);
        cudaFree(m->hb64);
        cudaFree(m->bb64);
        delete m;
    }
    ctx_release(ctx);
}

void isb_model_destroy(isb_model *m) { model_release(m); }

int isb_model_effective_couplings(isb_model *m, double *W, int64_t ld) {
    if (!m) return ISB_ERR_ARG;
    isb_ctx *ctx = m->ctx;
    ISB_LOCK(ctx);
    if (m->kind != ISB_KIND_BIPARTITE) return fail(ctx, ISB_ERR_STATE, "isb_model_effective_couplings: not a bipartite model");
    if (!W) return fail(ctx, ISB_ERR_ARG, "isb_model_effective_couplings: W is NULL");
    if (ld < m->nv) return fail(ctx, ISB_ERR_SIZE, "isb_model_effective_couplings: leading dimension %lld < nv = %d", (long long)ld, m->nv);
    ISB_CUDA(ctx, cudaSetDevice(ctx->device));
    std::vector<double> Wr((size_t)m->nv * m->nh);
    if (m->tc)
        ISB_TRY(isb::bip_tc_effective_couplings(m, Wr.data()));
    else
        ISB_CUDA(ctx, cudaMemcpy(Wr.data(), m->W64, Wr.size() * sizeof(double), cudaMemcpyDeviceToHost));
    for (int j = 0; j < m->nh; ++j)
        for (int i = 0; i < m->nv; ++i) W[i + (int64_t)j * ld] = Wr[(size_t)i * m->nh + j];
    return ISB_OK;
}

static bool general_graph(const isb_model *m) { return m->kind == ISB_KIND_DENSE || m->kind == ISB_KIND_SPARSE; }
int isb_model_num_visible(const isb_model *m) { return !m ? 0 : (general_graph(m) ? m->n : m->nv); }
int isb_model_num_hidden(const isb_model *m) { return !m ? 0 : (general_graph(m) ? 0 : m->nh); }
int isb_model_shard_block(const isb_model *m) { return !m ? 0 : m->shard_nb; }

// ------------------------------------------------------------------ ensembles
int isb_ens_create(isb_model *m, int R, isb_ens **out) {
    if (!m) return ISB_ERR_ARG;
    isb_ctx *ctx = m->ctx;
    ISB_LOCK(ctx);
    if (!out) return fail(ctx, ISB_ERR_ARG, "isb_ens_create: out is NULL");
    *out = nullptr;
    if (R <= 0) return fail(ctx, ISB_ERR_SIZE, "isb_ens_create: R = %d must be positive", R);
    if (m->kind == ISB_KIND_SHARD)
        return fail(ctx, ISB_ERR_STATE, "isb_ens_create: row-sharded models keep their spin matrices in caller-owned device buffers (isb_shard_halfstep_dev)");
    ISB_CUDA(ctx, cudaSetDevice(ctx->device));
    isb_ens *e = new isb_ens();
    e->model = m;
    m->refs.fetch_add(1);
    e->R = R;
    int rc = ISB_OK;
    do {
        cudaError_t ce;
        if (general_graph(m)) {
            e->lds = m->npad;
            ce = cudaMalloc(&e->spins, (size_t)R * e->lds);
            if (ce == cudaSuccess) ce = cudaMemsetAsync(e->spins, 1, (size_t)R * e->lds, ctx->stream);
            if (ce == cudaSuccess)
                ce = cudaMalloc(&e->fields, (size_t)R * m->npad * (m->fast_ok ? isb::ssf_field_elem_size(m) : sizeof(double)));
        } else {
            e->lds = (m->nv + 15) / 16 * 16;
            e->ldh = (m->nh + 15) / 16 * 16;
            ce = cudaMalloc(&e->spins, (size_t)R * e->lds);
            if (ce == cudaSuccess) ce = cudaMalloc(&e->hidden, (size_t)R * e->ldh);
            if (ce == cudaSuccess) ce = cudaMemsetAsync(e->spins, 1, (size_t)R * e->lds, ctx->stream);
            if (ce == cudaSuccess) ce = cudaMemsetAsync(e->hidden, 1, (size_t)R * e->ldh, ctx->stream);
        }
        if (ce == cudaSuccess) ce = cudaMalloc(&e->d_flips, (size_t)R * sizeof(unsigned long long));
        if (ce == cudaSuccess) ce = cudaMalloc(&e->d_counters, 4 * sizeof(unsigned long long));
        if (ce == cudaSuccess) ce = cudaMemsetAsync(e->d_counters, 0, 4 * sizeof(unsigned long long), ctx->stream);
        if (ce == cudaSuccess) ce = cudaStreamSynchronize(ctx->stream);
        if (ce != cudaSuccess) {
            rc = fail(ctx, ISB_ERR_CUDA, "isb_ens_create: allocation failed: %s", cudaGetErrorString(ce));
            break;
        }
        if (m->kind == ISB_KIND_BIPARTITE && m->prec != ISB_PREC_F64) rc = isb::bip_tc_ens_init(e);
    } while (0);
    if (rc) {
        isb_ens_destroy(e);
        return rc;
    }
    *out = e;
    return ISB_OK;
}

void isb_ens_destroy(isb_ens *e) {
    if (!e) return;
    isb_model *m = e->model;
    {
        ISB_LOCK(m->ctx);
        cudaSetDevice(m->ctx->device);
        cudaStreamSynchronize(m->ctx->stream);
        if (e->tc) isb::bip_tc_ens_free(e);
        cudaFree(e->spins);
        cudaFree(e->hidden);
        cudaFree(e->fields);
        cudaFree(e->ifields);
        cudaFree(e->spins2);
        cudaFree(e->fields2);
        cudaFree(e->ifields2);
        cudaFree(e->d_flips);
        cudaFree(e->d_counters);
        cudaFree(e->d_tscale);
        delete e;
    }
    model_release(m);
}

int isb_ens_replicas(const isb_ens *e) { return e ? e->R : 0; }

int isb_model_retain(isb_model *m) {
    if (!m) return ISB_ERR_ARG;
    m->refs.fetch_add(1);
    return ISB_OK;
}

int isb_ens_clone(isb_ens *src, isb_ens **out) {
    if (!src) return ISB_ERR_ARG;
    isb_ctx *ctx = src->model->ctx;
    ISB_LOCK(ctx);
    if (!out) return fail(ctx, ISB_ERR_ARG, "isb_ens_clone: out is NULL");
    *out = nullptr;
    isb_ens *e = nullptr;
    ISB_TRY(isb_ens_create(src->model, src->R, &e));
    cudaError_t ce = cudaSuccess;
    if (e->lds != src->lds || e->ldh != src->ldh) {
        isb_ens_destroy(e);
        return fail(ctx, ISB_ERR_STATE, "isb_ens_clone: layout mismatch");
    }
    ce = cudaMemcpyAsync(e->spins, src->spins, (size_t)src->R * src->lds, cudaMemcpyDeviceToDevice, ctx->stream);
    if (ce == cudaSuccess && src->hidden)
        ce = cudaMemcpyAsync(e->hidden, src->hidden, (size_t)src->R * src->ldh, cudaMemcpyDeviceToDevice, ctx->stream);
    if (ce == cudaSuccess && src->d_tscale) {
        ce = cudaMalloc(&e->d_tscale, (size_t)src->R * sizeof(double));
        if (ce == cudaSuccess)
            ce = cudaMemcpyAsync(e->d_tscale, src->d_tscale, (size_t)src->R * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream);
    }
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(ctx->stream);
    if (ce != cudaSuccess) {
        isb_ens_destroy(e);
        return fail(ctx, ISB_ERR_CUDA, "isb_ens_clone: copy failed: %s", cudaGetErrorString(ce));
    }
    e->tie_eps = src->tie_eps;
    e->fields_rule_sign = 0;  // the cached local fields are rebuilt from the copied spins by the next run
    *out = e;
    return ISB_OK;
}

static int copy_spins_in(isb_ens *e, int8_t *dst, int64_t ldd, int n, const int8_t *s, int64_t ld, const char *who) {
    isb_ctx *ctx = e->model->ctx;
    ISB_LOCK(ctx);
    if (!s) return fail(ctx, ISB_ERR_ARG, "%s: NULL spin array", who);
    if (ld < n) return fail(ctx, ISB_ERR_SIZE, "%s: leading dimension %lld < %d units", who, (long long)ld, n);
    for (int r = 0; r < e->R; ++r) {
        const int8_t *row = s + (int64_t)r * ld;
        unsigned bad = 0;  // branch-free so that the host compiler vectorises the scan
        for (int i = 0; i < n; ++i) bad |= (unsigned)((row[i] != 1) & (row[i] != -1));
        if (bad)
            for (int i = 0; i < n; ++i)
                if (row[i] != 1 && row[i] != -1)
                    return fail(ctx, ISB_ERR_ARG, "%s: spin [%d, replica %d] = %d is not +1 / -1", who, i, r, (int)row[i]);
    }
    ISB_CUDA(ctx, cudaSetDevice(ctx->device));
    ISB_CUDA(ctx, cudaMemcpy2DAsync(dst, (size_t)ldd, s, (size_t)ld, (size_t)n, (size_t)e->R, cudaMemcpyHostToDevice,
                                    ctx->stream));
    ISB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    e->fields_rule_sign = 0;
    e->ifields_ok = false;
    return ISB_OK;
}
static int copy_spins_out(isb_ens *e, const int8_t *src, int64_t lds, int n, int8_t *s, int64_t ld, const char *who) {
    isb_ctx *ctx = e->model->ctx;
    ISB_LOCK(ctx);
    if (!s) return fail(ctx, ISB_ERR_ARG, "%s: NULL spin array", who);
    if (ld < n) return fail(ctx, ISB_ERR_SIZE, "%s: leading dimension %lld < %d units", who, (long long)ld, n);
    ISB_CUDA(ctx, cudaSetDevice(ctx->device));
    ISB_CUDA(ctx, cudaMemcpy2DAsync(s, (size_t)ld, src, (size_t)lds, (size_t)n, (size_t)e->R, cudaMemcpyDeviceToHost,
                                    ctx->stream));
    ISB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return ISB_OK;
}

int isb_ens_set_spins(isb_ens *e, const int8_t *s, int64_t ld) {
    if (!e) return ISB_ERR_ARG;
    const isb_model *m = e->model;
    return copy_spins_in(e, e->spins, e->lds, general_graph(m) ? m->n : m->nv, s, ld, "isb_ens_set_spins");
}
int isb_ens_get_spins(isb_ens *e, int8_t *s, int64_t ld) {
    if (!e) return ISB_ERR_ARG;
    const isb_model *m = e->model;
    return copy_spins_out(e, e->spins, e->lds, general_graph(m) ? m->n : m->nv, s, ld, "isb_ens_get_spins");
}
int isb_ens_set_hidden(isb_ens *e, const int8_t *t, int64_t ld) {
    if (!e) return ISB_ERR_ARG;
    if (e->model->kind != ISB_KIND_BIPARTITE) return fail(e->model->ctx, ISB_ERR_STATE, "isb_ens_set_hidden: not a bipartite ensemble");
    return copy_spins_in(e, e->hidden, e->ldh, e->model->nh, t, ld, "isb_ens_set_hidden");
}
int isb_ens_get_hidden(isb_ens *e, int8_t *t, int64_t ld) {
    if (!e) return ISB_ERR_ARG;
    if (e->model->kind != ISB_KIND_BIPARTITE) return fail(e->model->ctx, ISB_ERR_STATE, "isb_ens_get_hidden: not a bipartite ensemble");
    return copy_spins_out(e, e->hidden, e->ldh, e->model->nh, t, ld, "isb_ens_get_hidden");
}

int isb_ens_energy(isb_ens *e, double *E) {
    if (!e) return ISB_ERR_ARG;
    isb_ctx *ctx = e->model->ctx;
    ISB_LOCK(ctx);
    if (!E) return fail(ctx, ISB_ERR_ARG, "isb_ens_energy: E is NULL");
    ISB_CUDA(ctx, cudaSetDevice(ctx->device));
    double *dE;
    ISB_TRY(isb::dev_reserve(ctx, isb::SCR_OUT, (size_t)e->R * sizeof(double), (void **)&dE));
    ISB_TRY(e->model->kind == ISB_KIND_DENSE    ? isb::dense_energy_device(e, dE)
            : e->model->kind == ISB_KIND_SPARSE ? isb::sparse_energy_device(e, dE)
                                                : isb::bip_energy_device(e, dE));
    ISB_TRY(d2h(ctx, E, dE, (size_t)e->R * sizeof(double), nullptr));
    ISB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return ISB_OK;
}

int isb_ens_magnetization(isb_ens *e, double *M) {
    if (!e) return ISB_ERR_ARG;
    isb_ctx *ctx = e->model->ctx;
    ISB_LOCK(ctx);
    if (!M) return fail(ctx, ISB_ERR_ARG, "isb_ens_magnetization: M is NULL");
    ISB_CUDA(ctx, cudaSetDevice(ctx->device));
    double *dM;
    ISB_TRY(isb::dev_reserve(ctx, isb::SCR_OUT, (size_t)e->R * sizeof(double), (void **)&dM));
    ISB_TRY(isb::magnetization_device(e, dM));
    ISB_TRY(d2h(ctx, M, dM, (size_t)e->R * sizeof(double), nullptr));
    ISB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return ISB_OK;
}

static int field_common(isb_ens *e, int layer, double *F, int64_t ld, const char *who) {
    isb_model *m = e->model;
    isb_ctx *ctx = m->ctx;
    ISB_LOCK(ctx);
    const int nout = general_graph(m) ? m->n : (layer == 0 ? m->nv : m->nh);
    if (!F) return fail(ctx, ISB_ERR_ARG, "%s: output is NULL", who);
    if (ld < nout) return fail(ctx, ISB_ERR_SIZE, "%s: leading dimension %lld < %d", who, (long long)ld, nout);
    ISB_CUDA(ctx, cudaSetDevice(ctx->device));
    double *dF;
    ISB_TRY(isb::dev_reserve(ctx, isb::SCR_OUT, (size_t)e->R * nout * sizeof(double), (void **)&dF));
    if (m->kind == ISB_KIND_DENSE)
        ISB_TRY(isb::dense_field_device(e, dF, nout));
    else if (m->kind == ISB_KIND_SPARSE)
        ISB_TRY(isb::sparse_field_device(e, dF, nout, nout, 1.0));
    else
        ISB_TRY(isb::bip_field_device(e, layer, dF, nout));
    ISB_CUDA(ctx, cudaMemcpy2DAsync(F, (size_t)ld * sizeof(double), dF, (size_t)nout * sizeof(double),
                                    (size_t)nout * sizeof(double), (size_t)e->R, cudaMemcpyDeviceToHost, ctx->stream));
    ISB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return ISB_OK;
}
int isb_ens_local_field(isb_ens *e, double *F, int64_t ld) {
    if (!e) return ISB_ERR_ARG;
    return field_common(e, 0, F, ld, "isb_ens_local_field");
}
int isb_ens_local_aux_bias(isb_ens *e, double *A, int64_t ld) {
    if (!e) return ISB_ERR_ARG;
    if (e->model->kind != ISB_KIND_BIPARTITE)
        return fail(e->model->ctx, ISB_ERR_STATE, "isb_ens_local_aux_bias: not a bipartite ensemble");
    return field_common(e, 1, A, ld, "isb_ens_local_aux_bias");
}

// ------------------------------------------------------------------ runs
static int check_schedule(isb_ctx *ctx, const char *who, const double *Tsched, int64_t nT, int64_t steps_per_T,
                          int64_t nsteps) {
    if (!Tsched || nT <= 0) return fail(ctx, ISB_ERR_ARG, "%s: a temperature schedule is required", who);
    if (steps_per_T <= 0) return fail(ctx, ISB_ERR_ARG, "%s: steps_per_T must be positive", who);
    if ((nsteps + steps_per_T - 1) / steps_per_T > nT)
        return fail(ctx, ISB_ERR_SIZE, "%s: schedule of %lld entries x %lld steps is shorter than %lld steps", who,
                    (long long)nT, (long long)steps_per_T, (long long)nsteps);
    if (!all_finite(Tsched, (size_t)nT)) return fail(ctx, ISB_ERR_NONFINITE, "%s: non-finite temperature", who);
    return ISB_OK;
}

static void begin_stats(isb_ens *e) {
    e->last_ms = 0.0;
    e->last_launches = e->last_h2d = e->last_d2h = 0;
    e->last_flips = e->last_near_ties = e->last_exact_fallbacks = 0;
}

// The end of a timed run, once ev1 follows its work and the copies of its results are queued: waits for them, reports a
// failed kernel, and puts the time from ev0 to ev1 into last_ms.
static int finish_run(isb_ens *e, const char *who) {
    isb_ctx *ctx = e->model->ctx;
    cudaError_t ce = cudaStreamSynchronize(ctx->stream);
    if (ce != cudaSuccess) return fail(ctx, ISB_ERR_CUDA, "%s: kernel failed: %s", who, cudaGetErrorString(ce));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
    e->last_ms = ms;
    return ISB_OK;
}

// finish_run of a single-spin run, which also reads back its flip counts per replica (d_flips [R]: into last_flips, and
// into out_flips when given) and its near-tie and exact-fallback counters.
static int finish_ssf_run(isb_ens *e, const char *who, const unsigned long long *d_flips, int64_t *out_flips) {
    isb_ctx *ctx = e->model->ctx;
    std::vector<unsigned long long> fl((size_t)e->R);
    unsigned long long counters[4] = {0, 0, 0, 0};
    ISB_TRY(d2h(ctx, fl.data(), d_flips, fl.size() * sizeof(unsigned long long), &e->last_d2h));
    ISB_TRY(d2h(ctx, counters, e->d_counters, sizeof counters, &e->last_d2h));
    ISB_TRY(finish_run(e, who));
    for (int r = 0; r < e->R; ++r) {
        e->last_flips += (int64_t)fl[r];
        if (out_flips) out_flips[r] = (int64_t)fl[r];
    }
    e->last_near_ties = (int64_t)counters[0];
    e->last_exact_fallbacks = (int64_t)counters[1];
    return ISB_OK;
}

// The checks every single-spin entry point shares: a general-graph ensemble, a known order (ISB_ORDER_CHECKERBOARD only on
// a periodic lattice) and, for the orders that walk the sites from `start`, start in [0, n).
static int check_ssf_run(isb_ens *e, const char *who, int order, int start) {
    const isb_model *m = e->model;
    isb_ctx *ctx = m->ctx;
    if (!general_graph(m)) return fail(ctx, ISB_ERR_STATE, "%s: not a general-graph ensemble", who);
    if (order < ISB_ORDER_SEQUENTIAL || order > ISB_ORDER_CHECKERBOARD) return fail(ctx, ISB_ERR_ARG, "%s: unknown order %d", who, order);
    if (order == ISB_ORDER_CHECKERBOARD && !isb::sparse_model_lattice(m))
        return fail(ctx, ISB_ERR_UNSUPPORTED,
                    "%s: ISB_ORDER_CHECKERBOARD needs a periodic L x L lattice (L a multiple of 32) with four neighbours per site", who);
    if ((order == ISB_ORDER_SEQUENTIAL || order == ISB_ORDER_CHECKERBOARD) && (start < 0 || start >= m->n))
        return fail(ctx, ISB_ERR_ARG, "%s: start = %d outside [0, %d)", who, start, m->n);
    return ISB_OK;
}

static int ssf_run_impl(isb_ens *e, int rule, int64_t nsteps, int order, const int32_t *nodes, int start, int fluct_mode,
                        const double *fluct, uint64_t seed, uint64_t step_offset, const double *Tsched, int64_t nT,
                        int64_t steps_per_T, int64_t trace_every, double *out_E, double *out_M, int64_t *out_flips,
                        int8_t *out_S, int64_t ldS, int64_t *hist);

int isb_ssf_run(isb_ens *e, int rule, int64_t nsteps, int order, const int32_t *nodes, int start, int fluct_mode,
                const double *fluct, uint64_t seed, uint64_t step_offset, const double *Tsched, int64_t nT,
                int64_t steps_per_T, int64_t trace_every, double *out_E, double *out_M, int64_t *out_flips) {
    return ssf_run_impl(e, rule, nsteps, order, nodes, start, fluct_mode, fluct, seed, step_offset, Tsched, nT,
                        steps_per_T, trace_every, out_E, out_M, out_flips, nullptr, 0, nullptr);
}

int isb_ssf_run_snap(isb_ens *e, int rule, int64_t nsteps, int order, const int32_t *nodes, int start, int fluct_mode,
                     const double *fluct, uint64_t seed, uint64_t step_offset, const double *Tsched, int64_t nT,
                     int64_t steps_per_T, int64_t trace_every, double *out_E, double *out_M, int64_t *out_flips,
                     int8_t *out_S, int64_t ldS) {
    return ssf_run_impl(e, rule, nsteps, order, nodes, start, fluct_mode, fluct, seed, step_offset, Tsched, nT,
                        steps_per_T, trace_every, out_E, out_M, out_flips, out_S, ldS, nullptr);
}

int isb_ssf_run_hist(isb_ens *e, int rule, int64_t nsteps, int order, const int32_t *nodes, int start, int fluct_mode,
                     const double *fluct, uint64_t seed, uint64_t step_offset, const double *Tsched, int64_t nT,
                     int64_t steps_per_T, int64_t trace_every, int64_t *hist) {
    if (!e) return ISB_ERR_ARG;
    isb_ctx *ctx = e->model->ctx;
    ISB_LOCK(ctx);
    if (!hist) return fail(ctx, ISB_ERR_ARG, "isb_ssf_run_hist: hist is NULL");
    if (general_graph(e->model) && e->model->n > 24)
        return fail(ctx, ISB_ERR_SIZE, "isb_ssf_run_hist: N = %d > 24 (the histogram has 2^N bins)", e->model->n);
    if (trace_every <= 0) return fail(ctx, ISB_ERR_ARG, "isb_ssf_run_hist: trace_every must be positive");
    return ssf_run_impl(e, rule, nsteps, order, nodes, start, fluct_mode, fluct, seed, step_offset, Tsched, nT,
                        steps_per_T, trace_every, nullptr, nullptr, nullptr, nullptr, 0, hist);
}

static int ssf_run_impl(isb_ens *e, int rule, int64_t nsteps, int order, const int32_t *nodes, int start, int fluct_mode,
                        const double *fluct, uint64_t seed, uint64_t step_offset, const double *Tsched, int64_t nT,
                        int64_t steps_per_T, int64_t trace_every, double *out_E, double *out_M, int64_t *out_flips,
                        int8_t *out_S, int64_t ldS, int64_t *hist) {
    if (!e) return ISB_ERR_ARG;
    isb_model *m = e->model;
    isb_ctx *ctx = m->ctx;
    ISB_LOCK(ctx);
    const char *who = "isb_ssf_run";
    ISB_TRY(check_ssf_run(e, who, order, start));
    if (rule < ISB_RULE_HOPFIELD || rule > ISB_RULE_METROPOLIS) return fail(ctx, ISB_ERR_ARG, "%s: unknown rule %d", who, rule);
    if (nsteps < 0) return fail(ctx, ISB_ERR_ARG, "%s: nsteps = %lld is negative", who, (long long)nsteps);
    if (fluct_mode < ISB_FLUCT_PHILOX || fluct_mode > ISB_FLUCT_PER_REPLICA)
        return fail(ctx, ISB_ERR_ARG, "%s: unknown fluct_mode %d", who, fluct_mode);
    if (trace_every < 0) return fail(ctx, ISB_ERR_ARG, "%s: trace_every is negative", who);
    if (out_S && ldS < m->n) return fail(ctx, ISB_ERR_SIZE, "%s: snapshot pitch %lld < N = %d", who, (long long)ldS, m->n);
    const bool stochastic = rule != ISB_RULE_HOPFIELD;
    if (!stochastic) fluct_mode = ISB_FLUCT_PHILOX;  // the fluctuation is a dummy (SingleSpinFlip.jl:31)
    if (order == ISB_ORDER_LIST) {
        if (!nodes && nsteps > 0) return fail(ctx, ISB_ERR_ARG, "%s: ISB_ORDER_LIST needs a node list", who);
        for (int64_t k = 0; k < nsteps; ++k)
            if (nodes[k] < 0 || nodes[k] >= m->n)
                return fail(ctx, ISB_ERR_ARG, "%s: nodes[%lld] = %d outside [0, %d)", who, (long long)k, nodes[k], m->n);
    }
    if (fluct_mode != ISB_FLUCT_PHILOX) {
        if (!fluct && nsteps > 0) return fail(ctx, ISB_ERR_ARG, "%s: fluctuation array is NULL", who);
        const size_t nf = (size_t)nsteps * (fluct_mode == ISB_FLUCT_PER_REPLICA ? (size_t)e->R : 1);
        if (!all_finite(fluct, nf)) return fail(ctx, ISB_ERR_NONFINITE, "%s: non-finite fluctuation", who);
    }
    const double zeroT = 0.0;
    if (stochastic) {
        ISB_TRY(check_schedule(ctx, who, Tsched, nT, steps_per_T, nsteps));
    } else {
        Tsched = &zeroT;
        nT = 1;
        steps_per_T = std::max<int64_t>(nsteps, 1);
    }
    ISB_CUDA(ctx, cudaSetDevice(ctx->device));
    begin_stats(e);
    if (nsteps == 0) {
        if (out_flips) std::fill(out_flips, out_flips + e->R, (int64_t)0);
        return ISB_OK;
    }

    int32_t *d_nodes = nullptr;
    double *d_fluct = nullptr, *d_T = nullptr, *d_E = nullptr, *d_M = nullptr;
    if (order == ISB_ORDER_LIST || order == ISB_ORDER_RANDOM) {
        ISB_TRY(isb::dev_reserve(ctx, isb::SCR_NODES, (size_t)nsteps * sizeof(int32_t), (void **)&d_nodes));
        if (order == ISB_ORDER_LIST)
            ISB_TRY(h2d(ctx, d_nodes, nodes, (size_t)nsteps * sizeof(int32_t), &e->last_h2d));
    }
    if (fluct_mode != ISB_FLUCT_PHILOX) {
        const size_t nf = (size_t)nsteps * (fluct_mode == ISB_FLUCT_PER_REPLICA ? (size_t)e->R : 1);
        ISB_TRY(isb::dev_reserve(ctx, isb::SCR_FLUCT, nf * sizeof(double), (void **)&d_fluct));
        ISB_TRY(h2d(ctx, d_fluct, fluct, nf * sizeof(double), &e->last_h2d));
    }
    ISB_TRY(isb::dev_reserve(ctx, isb::SCR_T, (size_t)nT * sizeof(double), (void **)&d_T));
    ISB_TRY(h2d(ctx, d_T, Tsched, (size_t)nT * sizeof(double), &e->last_h2d));
    const int64_t ntr = trace_every > 0 ? nsteps / trace_every : 0;
    if (ntr > 0 && out_E) ISB_TRY(isb::dev_reserve(ctx, isb::SCR_E, (size_t)ntr * e->R * sizeof(double), (void **)&d_E));
    if (ntr > 0 && out_M) ISB_TRY(isb::dev_reserve(ctx, isb::SCR_M, (size_t)ntr * e->R * sizeof(double), (void **)&d_M));
    int8_t *d_S = nullptr;
    if (ntr > 0 && (out_S || hist)) ISB_TRY(isb::dev_reserve(ctx, isb::SCR_S, (size_t)ntr * e->R * m->n, (void **)&d_S));
    unsigned long long *d_hist = nullptr;
    if (d_S && hist) {
        ISB_TRY(isb::dev_reserve(ctx, isb::SCR_HIST, sizeof(unsigned long long) << m->n, (void **)&d_hist));
        ISB_CUDA(ctx, cudaMemsetAsync(d_hist, 0, sizeof(unsigned long long) << m->n, ctx->stream));
    }
    ISB_CUDA(ctx, cudaMemsetAsync(e->d_counters, 0, 4 * sizeof(unsigned long long), ctx->stream));

    ISB_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    ISB_TRY(isb::ssf_sweep_device(e, rule, nsteps, order, d_nodes, start, fluct_mode, d_fluct, seed, step_offset, d_T,
                                  steps_per_T, (d_E || d_M || d_S) ? trace_every : 0, d_E, d_M, d_S));
    if (d_hist) {
        ISB_TRY(isb::config_histogram_device(ctx, d_S, ntr * e->R, m->n, d_hist));
        e->last_launches += 1;
    }
    ISB_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));

    std::vector<unsigned long long> hh;
    if (d_hist) {
        hh.resize((size_t)1 << m->n);
        ISB_TRY(d2h(ctx, hh.data(), d_hist, hh.size() * sizeof(unsigned long long), &e->last_d2h));
    }
    if (d_E) ISB_TRY(d2h(ctx, out_E, d_E, (size_t)ntr * e->R * sizeof(double), &e->last_d2h));
    if (d_M) ISB_TRY(d2h(ctx, out_M, d_M, (size_t)ntr * e->R * sizeof(double), &e->last_d2h));
    if (d_S && out_S) {
        ISB_CUDA(ctx, cudaMemcpy2DAsync(out_S, (size_t)ldS, d_S, (size_t)m->n, (size_t)m->n, (size_t)ntr * e->R,
                                        cudaMemcpyDeviceToHost, ctx->stream));
        e->last_d2h += (int64_t)ntr * e->R * m->n;
    }
    ISB_TRY(finish_ssf_run(e, who, e->d_flips, out_flips));
    for (size_t b = 0; b < hh.size(); ++b) hist[b] += (int64_t)hh[b];
    return ISB_OK;
}

int isb_ssf_run_pt(isb_ens *e, int rule, int n_levels, const double *levels, int64_t rounds, int64_t steps_per_round,
                   int order, int start, uint64_t seed, uint64_t step_offset, uint64_t round_offset, int32_t *level_of,
                   double *out_E, double *out_M, double *out_Q, int64_t *out_accepted, int64_t *out_flips) {
    if (!e) return ISB_ERR_ARG;
    isb_model *m = e->model;
    isb_ctx *ctx = m->ctx;
    ISB_LOCK(ctx);
    const char *who = "isb_ssf_run_pt";
    ISB_TRY(check_ssf_run(e, who, order, start));
    if (rule != ISB_RULE_GLAUBER && rule != ISB_RULE_METROPOLIS)
        return fail(ctx, ISB_ERR_ARG, "%s: rule %d has no temperature to exchange (Glauber or Metropolis only)", who, rule);
    if (order == ISB_ORDER_LIST) return fail(ctx, ISB_ERR_ARG, "%s: order %d is not sequential, random or checkerboard", who, order);
    if (n_levels < 1) return fail(ctx, ISB_ERR_ARG, "%s: n_levels = %d must be positive", who, n_levels);
    if (n_levels > 1024) return fail(ctx, ISB_ERR_UNSUPPORTED, "%s: n_levels = %d > 1024", who, n_levels);
    if (e->R % n_levels != 0)
        return fail(ctx, ISB_ERR_SIZE, "%s: R = %d replicas is not a multiple of n_levels = %d", who, e->R, n_levels);
    const int L = n_levels, G = e->R / n_levels;
    if (!levels || !level_of) return fail(ctx, ISB_ERR_ARG, "%s: levels and level_of are required", who);
    if (!all_finite(levels, (size_t)L)) return fail(ctx, ISB_ERR_NONFINITE, "%s: non-finite temperature level", who);
    for (int l = 0; l < L; ++l)
        if (!(levels[l] > 0.0)) return fail(ctx, ISB_ERR_ARG, "%s: levels[%d] = %g must be positive", who, l, levels[l]);
    {
        std::vector<char> seen((size_t)L);
        for (int g = 0; g < G; ++g) {
            std::fill(seen.begin(), seen.end(), 0);
            for (int s = 0; s < L; ++s) {
                const int32_t v = level_of[(size_t)g * L + s];
                if (v < 0 || v >= L || seen[v])
                    return fail(ctx, ISB_ERR_ARG, "%s: level_of of ladder %d is not a permutation of 0..%d", who, g, L - 1);
                seen[v] = 1;
            }
        }
    }
    if (out_Q && G % 2 != 0) return fail(ctx, ISB_ERR_SIZE, "%s: overlaps pair ladders 2p, 2p+1; %d ladders is odd", who, G);
    if (steps_per_round <= 0)
        return fail(ctx, ISB_ERR_ARG, "%s: steps_per_round = %lld must be positive", who, (long long)steps_per_round);
    if (rounds < 0) return fail(ctx, ISB_ERR_ARG, "%s: rounds = %lld is negative", who, (long long)rounds);
    ISB_CUDA(ctx, cudaSetDevice(ctx->device));
    begin_stats(e);
    if (out_accepted) std::fill(out_accepted, out_accepted + (L - 1), (int64_t)0);
    if (rounds == 0) {
        if (out_flips) std::fill(out_flips, out_flips + e->R, (int64_t)0);
        return ISB_OK;
    }

    // device state of the call: levels [L] | accepted [L] | flip totals [R] (8-byte words) | level_of [R] (int32)
    const size_t R = (size_t)e->R;
    char *st = nullptr;
    ISB_TRY(isb::dev_reserve(ctx, isb::SCR_PT_STATE, 8 * (2 * (size_t)L + R) + 4 * R, (void **)&st));
    double *d_levels = (double *)st;
    unsigned long long *d_acc = (unsigned long long *)(st + 8 * (size_t)L);
    unsigned long long *d_ftot = (unsigned long long *)(st + 16 * (size_t)L);
    int32_t *d_level_of = (int32_t *)(st + 8 * (2 * (size_t)L + R));
    int32_t *d_nodes = nullptr;
    double *d_T = nullptr, *d_Er = nullptr, *d_Mr = nullptr, *d_recE = nullptr, *d_recM = nullptr, *d_recQ = nullptr;
    if (order == ISB_ORDER_RANDOM)
        ISB_TRY(isb::dev_reserve(ctx, isb::SCR_NODES, (size_t)steps_per_round * sizeof(int32_t), (void **)&d_nodes));
    ISB_TRY(isb::dev_reserve(ctx, isb::SCR_T, sizeof(double), (void **)&d_T));
    ISB_TRY(isb::dev_reserve(ctx, isb::SCR_E, R * sizeof(double), (void **)&d_Er));
    if (out_M) ISB_TRY(isb::dev_reserve(ctx, isb::SCR_M, R * sizeof(double), (void **)&d_Mr));
    if (out_E) ISB_TRY(isb::dev_reserve(ctx, isb::SCR_PT_E, (size_t)rounds * R * sizeof(double), (void **)&d_recE));
    if (out_M) ISB_TRY(isb::dev_reserve(ctx, isb::SCR_PT_M, (size_t)rounds * R * sizeof(double), (void **)&d_recM));
    if (out_Q) ISB_TRY(isb::dev_reserve(ctx, isb::SCR_PT_Q, (size_t)rounds * L * (G / 2) * sizeof(double), (void **)&d_recQ));
    if (!e->d_tscale) ISB_CUDA(ctx, cudaMalloc(&e->d_tscale, R * sizeof(double)));
    std::vector<double> tsc(R);
    for (size_t r = 0; r < R; ++r) tsc[r] = levels[level_of[r]];
    const double one = 1.0;
    ISB_TRY(h2d(ctx, d_levels, levels, (size_t)L * sizeof(double), &e->last_h2d));
    ISB_TRY(h2d(ctx, d_level_of, level_of, R * sizeof(int32_t), &e->last_h2d));
    ISB_TRY(h2d(ctx, e->d_tscale, tsc.data(), R * sizeof(double), &e->last_h2d));
    ISB_TRY(h2d(ctx, d_T, &one, sizeof(double), &e->last_h2d));
    ISB_CUDA(ctx, cudaMemsetAsync(d_acc, 0, 8 * ((size_t)L + R), ctx->stream));
    ISB_CUDA(ctx, cudaMemsetAsync(e->d_counters, 0, 4 * sizeof(unsigned long long), ctx->stream));

    ISB_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    ISB_TRY(isb::ssf_pt_run_device(e, rule, L, d_levels, rounds, steps_per_round, order, start, seed, step_offset,
                                   round_offset, d_nodes, d_T, d_level_of, d_Er, d_Mr, d_recE, d_recM, d_recQ, d_acc, d_ftot));
    ISB_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));

    std::vector<unsigned long long> acc((size_t)L);
    ISB_TRY(d2h(ctx, level_of, d_level_of, R * sizeof(int32_t), &e->last_d2h));
    ISB_TRY(d2h(ctx, acc.data(), d_acc, (size_t)L * sizeof(unsigned long long), &e->last_d2h));
    if (d_recE) ISB_TRY(d2h(ctx, out_E, d_recE, (size_t)rounds * R * sizeof(double), &e->last_d2h));
    if (d_recM) ISB_TRY(d2h(ctx, out_M, d_recM, (size_t)rounds * R * sizeof(double), &e->last_d2h));
    if (d_recQ) ISB_TRY(d2h(ctx, out_Q, d_recQ, (size_t)rounds * L * (G / 2) * sizeof(double), &e->last_d2h));
    ISB_TRY(finish_ssf_run(e, who, d_ftot, out_flips));
    if (out_accepted)
        for (int l = 0; l + 1 < L; ++l) out_accepted[l] = (int64_t)acc[l];
    return ISB_OK;
}

int isb_ens_select_replicas(isb_ens *e, const int32_t *src) {
    if (!e) return ISB_ERR_ARG;
    isb_ctx *ctx = e->model->ctx;
    ISB_LOCK(ctx);
    const char *who = "isb_ens_select_replicas";
    if (!general_graph(e->model)) return fail(ctx, ISB_ERR_STATE, "%s: not a general-graph ensemble", who);
    if (!src) return fail(ctx, ISB_ERR_ARG, "%s: src is NULL", who);
    for (int r = 0; r < e->R; ++r)
        if (src[r] < 0 || src[r] >= e->R)
            return fail(ctx, ISB_ERR_ARG, "%s: src[%d] = %d outside [0, %d)", who, r, src[r], e->R);
    ISB_CUDA(ctx, cudaSetDevice(ctx->device));
    begin_stats(e);
    int32_t *d_src = nullptr;
    ISB_TRY(isb::dev_reserve(ctx, isb::SCR_PA_STATE, (size_t)e->R * sizeof(int32_t), (void **)&d_src));
    ISB_TRY(h2d(ctx, d_src, src, (size_t)e->R * sizeof(int32_t), &e->last_h2d));
    ISB_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    ISB_TRY(isb::ens_select_device(e, d_src));
    ISB_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    return finish_run(e, who);
}

int isb_ssf_run_pa(isb_ens *e, int rule, int n_pop, int64_t nT, const double *T, double T_next, int64_t steps_per_T,
                   int order, int start, uint64_t seed, uint64_t step_offset, uint64_t T_offset, int32_t *family,
                   double *out_E, double *out_M, double *out_lnQ, int64_t *out_flips) {
    if (!e) return ISB_ERR_ARG;
    isb_model *m = e->model;
    isb_ctx *ctx = m->ctx;
    ISB_LOCK(ctx);
    const char *who = "isb_ssf_run_pa";
    ISB_TRY(check_ssf_run(e, who, order, start));
    if (rule != ISB_RULE_GLAUBER && rule != ISB_RULE_METROPOLIS)
        return fail(ctx, ISB_ERR_ARG, "%s: rule %d has no temperature to anneal (Glauber or Metropolis only)", who, rule);
    if (order == ISB_ORDER_LIST) return fail(ctx, ISB_ERR_ARG, "%s: order %d is not sequential, random or checkerboard", who, order);
    if (e->d_tscale)
        return fail(ctx, ISB_ERR_STATE, "%s: per-replica temperature factors are set (clear them first)", who);
    if (n_pop < 1) return fail(ctx, ISB_ERR_ARG, "%s: n_pop = %d must be positive", who, n_pop);
    if (e->R % n_pop != 0)
        return fail(ctx, ISB_ERR_SIZE, "%s: R = %d replicas is not a multiple of n_pop = %d", who, e->R, n_pop);
    const int P = e->R / n_pop;
    if (P > (1 << 20)) return fail(ctx, ISB_ERR_UNSUPPORTED, "%s: population size %d > 2^20", who, P);
    if (nT < 0) return fail(ctx, ISB_ERR_ARG, "%s: nT = %lld is negative", who, (long long)nT);
    if (nT > 0 && !T) return fail(ctx, ISB_ERR_ARG, "%s: T is NULL", who);
    if (!all_finite(T, (size_t)nT) || !std::isfinite(T_next))
        return fail(ctx, ISB_ERR_NONFINITE, "%s: non-finite temperature", who);
    for (int64_t k = 0; k < nT; ++k)
        if (!(T[k] > 0.0)) return fail(ctx, ISB_ERR_ARG, "%s: T[%lld] = %g must be positive", who, (long long)k, T[k]);
    if (T_next < 0.0) return fail(ctx, ISB_ERR_ARG, "%s: T_next = %g is negative (0: none)", who, T_next);
    if (steps_per_T <= 0)
        return fail(ctx, ISB_ERR_ARG, "%s: steps_per_T = %lld must be positive", who, (long long)steps_per_T);
    ISB_CUDA(ctx, cudaSetDevice(ctx->device));
    begin_stats(e);
    if (nT == 0) {
        if (out_flips) std::fill(out_flips, out_flips + e->R, (int64_t)0);
        return ISB_OK;
    }
    const int64_t n_res = nT - 1 + (T_next > 0.0 ? 1 : 0);
    std::vector<double> db((size_t)n_res);
    for (int64_t k = 0; k < n_res; ++k) db[k] = 1.0 / (k + 1 < nT ? T[k + 1] : T_next) - 1.0 / T[k];

    // device state of the call, 8-byte words: flip totals | C (CTA-local) | CTA sums of W | a | CTA maxima | CTA sums of
    // x [R each] | population maxima [n_pop] | E [R] | lnQ [n_res][n_pop]; then int32: parent | family x 2 [R each]
    const size_t R = (size_t)e->R, np = (size_t)n_pop;
    const size_t words = 7 * R + np + (size_t)n_res * np;
    char *st = nullptr;
    ISB_TRY(isb::dev_reserve(ctx, isb::SCR_PA_STATE, 8 * words + 4 * 3 * R, (void **)&st));
    isb::PaDevice d{};
    d.flips_total = (unsigned long long *)st;
    d.cloc = d.flips_total + R;
    d.bW = d.cloc + R;
    d.a = (double *)(d.bW + R);
    d.bmax = d.a + R;
    d.bx = d.bmax + R;
    d.pmax = d.bx + R;
    d.E = d.pmax + np;
    d.lnQ = d.E + R;
    d.parent = (int32_t *)(st + 8 * words);
    if (family) {
        d.fam[0] = d.parent + R;
        d.fam[1] = d.fam[0] + R;
    }
    double *d_T = nullptr;
    if (order == ISB_ORDER_RANDOM)
        ISB_TRY(isb::dev_reserve(ctx, isb::SCR_NODES, (size_t)steps_per_T * sizeof(int32_t), (void **)&d.nodes));
    ISB_TRY(isb::dev_reserve(ctx, isb::SCR_T, (size_t)nT * sizeof(double), (void **)&d_T));
    d.T = d_T;
    if (out_E) ISB_TRY(isb::dev_reserve(ctx, isb::SCR_E, (size_t)nT * R * sizeof(double), (void **)&d.recE));
    if (out_M) ISB_TRY(isb::dev_reserve(ctx, isb::SCR_M, (size_t)nT * R * sizeof(double), (void **)&d.recM));
    ISB_TRY(h2d(ctx, d_T, T, (size_t)nT * sizeof(double), &e->last_h2d));
    if (family) ISB_TRY(h2d(ctx, d.fam[0], family, R * sizeof(int32_t), &e->last_h2d));
    ISB_CUDA(ctx, cudaMemsetAsync(d.flips_total, 0, R * sizeof(unsigned long long), ctx->stream));
    ISB_CUDA(ctx, cudaMemsetAsync(e->d_counters, 0, 4 * sizeof(unsigned long long), ctx->stream));

    int fam_final = 0;
    ISB_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    ISB_TRY(isb::ssf_pa_run_device(e, rule, n_pop, nT, db.data(), n_res, steps_per_T, order, start, seed, step_offset,
                                   T_offset, d, &fam_final));
    ISB_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));

    if (family) ISB_TRY(d2h(ctx, family, d.fam[fam_final], R * sizeof(int32_t), &e->last_d2h));
    if (out_E) ISB_TRY(d2h(ctx, out_E, d.recE, (size_t)nT * R * sizeof(double), &e->last_d2h));
    if (out_M) ISB_TRY(d2h(ctx, out_M, d.recM, (size_t)nT * R * sizeof(double), &e->last_d2h));
    if (out_lnQ) ISB_TRY(d2h(ctx, out_lnQ, d.lnQ, (size_t)n_res * np * sizeof(double), &e->last_d2h));
    return finish_ssf_run(e, who, d.flips_total, out_flips);
}

int isb_philox_fluct(isb_ctx *ctx, int rule, int prec, uint64_t seed, uint64_t step_offset, int r0, int nr,
                     int64_t nsteps, double *out) {
    (void)prec;
    if (!ctx) return ISB_ERR_ARG;
    ISB_LOCK(ctx);
    if (!out || nr < 0 || nsteps < 0 || r0 < 0) return fail(ctx, ISB_ERR_ARG, "isb_philox_fluct: bad argument");
    ISB_CUDA(ctx, cudaSetDevice(ctx->device));
    double *d;
    const size_t bytes = (size_t)nr * nsteps * sizeof(double);
    ISB_TRY(isb::dev_reserve(ctx, isb::SCR_OUT, bytes, (void **)&d));
    ISB_TRY(isb::philox_fluct_device(ctx, rule, seed, step_offset, r0, nr, nsteps, d));
    ISB_TRY(d2h(ctx, out, d, bytes, nullptr));
    ISB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return ISB_OK;
}

int isb_philox_nodes(isb_ctx *ctx, int n, uint64_t seed, uint64_t step_offset, int64_t nsteps, int32_t *out) {
    if (!ctx) return ISB_ERR_ARG;
    ISB_LOCK(ctx);
    if (!out || n <= 0 || nsteps < 0) return fail(ctx, ISB_ERR_ARG, "isb_philox_nodes: bad argument");
    ISB_CUDA(ctx, cudaSetDevice(ctx->device));
    int32_t *d;
    ISB_TRY(isb::dev_reserve(ctx, isb::SCR_OUT, (size_t)nsteps * sizeof(int32_t), (void **)&d));
    ISB_TRY(isb::philox_nodes_device(ctx, n, seed, step_offset, nsteps, d));
    ISB_TRY(d2h(ctx, out, d, (size_t)nsteps * sizeof(int32_t), nullptr));
    ISB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return ISB_OK;
}

int isb_philox_raw(isb_ctx *ctx, const uint32_t *ctr, const uint32_t key[2], int nblocks, uint32_t *out) {
    if (!ctx) return ISB_ERR_ARG;
    ISB_LOCK(ctx);
    if (!ctr || !key || !out || nblocks < 0) return fail(ctx, ISB_ERR_ARG, "isb_philox_raw: bad argument");
    ISB_CUDA(ctx, cudaSetDevice(ctx->device));
    uint32_t *dc, *dout;
    const size_t bytes = (size_t)nblocks * 4 * sizeof(uint32_t);
    ISB_TRY(isb::dev_reserve(ctx, isb::SCR_TMP, bytes, (void **)&dc));
    ISB_TRY(isb::dev_reserve(ctx, isb::SCR_OUT, bytes, (void **)&dout));
    ISB_TRY(h2d(ctx, dc, ctr, bytes, nullptr));
    ISB_TRY(isb::philox_raw_device(ctx, dc, key[0], key[1], nblocks, dout));
    ISB_TRY(d2h(ctx, out, dout, bytes, nullptr));
    ISB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return ISB_OK;
}

int isb_bip_run(isb_ens *e, int rule, int64_t nsteps, int fluct_mode, const double *Fv, const double *Fh,
                uint64_t seed, uint64_t step_offset, const double *Tsched, int64_t nT, int64_t steps_per_T,
                int64_t trace_every, double *out_E) {
    return isb_bip_run_snap(e, rule, nsteps, fluct_mode, Fv, Fh, seed, step_offset, Tsched, nT, steps_per_T, trace_every,
                            out_E, nullptr, 0, nullptr, 0);
}

int isb_bip_run_snap(isb_ens *e, int rule, int64_t nsteps, int fluct_mode, const double *Fv, const double *Fh,
                     uint64_t seed, uint64_t step_offset, const double *Tsched, int64_t nT, int64_t steps_per_T,
                     int64_t trace_every, double *out_E, int8_t *out_Sv, int64_t ldSv, int8_t *out_Sh, int64_t ldSh) {
    if (!e) return ISB_ERR_ARG;
    isb_model *m = e->model;
    isb_ctx *ctx = m->ctx;
    ISB_LOCK(ctx);
    const char *who = "isb_bip_run";
    if (m->kind != ISB_KIND_BIPARTITE) return fail(ctx, ISB_ERR_STATE, "%s: not a bipartite ensemble", who);
    if (rule != ISB_BIP_SCA && rule != ISB_BIP_MA) return fail(ctx, ISB_ERR_ARG, "%s: unknown rule %d", who, rule);
    if (nsteps < 0) return fail(ctx, ISB_ERR_ARG, "%s: nsteps = %lld is negative", who, (long long)nsteps);
    if (fluct_mode < ISB_FLUCT_PHILOX || fluct_mode > ISB_FLUCT_PER_REPLICA)
        return fail(ctx, ISB_ERR_ARG, "%s: unknown fluct_mode %d", who, fluct_mode);
    if (trace_every < 0) return fail(ctx, ISB_ERR_ARG, "%s: trace_every is negative", who);
    ISB_TRY(check_schedule(ctx, who, Tsched, nT, steps_per_T, nsteps));
    const size_t rep = fluct_mode == ISB_FLUCT_PER_REPLICA ? (size_t)e->R : 1;
    const size_t nfv = (size_t)nsteps * m->nv * rep, nfh = (size_t)nsteps * m->nh * rep;
    if (fluct_mode != ISB_FLUCT_PHILOX && nsteps > 0) {
        if (!Fv || !Fh) return fail(ctx, ISB_ERR_ARG, "%s: fluctuation arrays are NULL", who);
        if (!all_finite(Fv, nfv) || !all_finite(Fh, nfh)) return fail(ctx, ISB_ERR_NONFINITE, "%s: non-finite fluctuation", who);
    }
    ISB_CUDA(ctx, cudaSetDevice(ctx->device));
    begin_stats(e);
    if (nsteps == 0) return ISB_OK;
    double *d_Fv = nullptr, *d_Fh = nullptr, *d_T = nullptr, *d_E = nullptr;
    if (fluct_mode != ISB_FLUCT_PHILOX) {
        ISB_TRY(isb::dev_reserve(ctx, isb::SCR_FLUCT, nfv * sizeof(double), (void **)&d_Fv));
        ISB_TRY(isb::dev_reserve(ctx, isb::SCR_FLUCT2, nfh * sizeof(double), (void **)&d_Fh));
        ISB_TRY(h2d(ctx, d_Fv, Fv, nfv * sizeof(double), &e->last_h2d));
        ISB_TRY(h2d(ctx, d_Fh, Fh, nfh * sizeof(double), &e->last_h2d));
    }
    ISB_TRY(isb::dev_reserve(ctx, isb::SCR_T, (size_t)nT * sizeof(double), (void **)&d_T));
    ISB_TRY(h2d(ctx, d_T, Tsched, (size_t)nT * sizeof(double), &e->last_h2d));
    if ((out_Sv && ldSv < m->nv) || (out_Sh && ldSh < m->nh)) return fail(ctx, ISB_ERR_SIZE, "%s: snapshot pitch too small", who);
    const int64_t ntr = (trace_every > 0 && (out_E || out_Sv || out_Sh)) ? nsteps / trace_every : 0;
    if (ntr > 0 && out_E) ISB_TRY(isb::dev_reserve(ctx, isb::SCR_E, (size_t)ntr * e->R * sizeof(double), (void **)&d_E));
    int8_t *d_Sv = nullptr, *d_Sh = nullptr;
    if (ntr > 0 && out_Sv) ISB_TRY(isb::dev_reserve(ctx, isb::SCR_S, (size_t)ntr * e->R * m->nv, (void **)&d_Sv));
    if (ntr > 0 && out_Sh) ISB_TRY(isb::dev_reserve(ctx, isb::SCR_S2, (size_t)ntr * e->R * m->nh, (void **)&d_Sh));

    ISB_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    if (m->prec == ISB_PREC_F64)
        ISB_TRY(isb::bip_run_exact_device(e, rule, nsteps, fluct_mode, d_Fv, d_Fh, seed, step_offset, d_T, steps_per_T,
                                          trace_every, d_E, d_Sv, d_Sh));
    else
        ISB_TRY(isb::bip_run_tc_device(e, rule, nsteps, fluct_mode, d_Fv, d_Fh, seed, step_offset, d_T, steps_per_T,
                                       trace_every, d_E, d_Sv, d_Sh));
    ISB_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    if (d_E) ISB_TRY(d2h(ctx, out_E, d_E, (size_t)ntr * e->R * sizeof(double), &e->last_d2h));
    if (d_Sv) {
        ISB_CUDA(ctx, cudaMemcpy2DAsync(out_Sv, (size_t)ldSv, d_Sv, (size_t)m->nv, (size_t)m->nv, (size_t)ntr * e->R,
                                        cudaMemcpyDeviceToHost, ctx->stream));
        e->last_d2h += ntr * e->R * m->nv;
    }
    if (d_Sh) {
        ISB_CUDA(ctx, cudaMemcpy2DAsync(out_Sh, (size_t)ldSh, d_Sh, (size_t)m->nh, (size_t)m->nh, (size_t)ntr * e->R,
                                        cudaMemcpyDeviceToHost, ctx->stream));
        e->last_d2h += ntr * e->R * m->nh;
    }
    return finish_run(e, who);
}

int isb_philox_bip_fluct(isb_ctx *ctx, int rule, int prec, uint64_t seed, uint64_t step_offset, int layer, int nunits,
                         int r0, int nr, int64_t nsteps, double *out) {
    (void)prec;
    if (!ctx) return ISB_ERR_ARG;
    ISB_LOCK(ctx);
    if (!out || nr < 0 || nsteps < 0 || r0 < 0 || nunits <= 0 || (layer != 0 && layer != 1))
        return fail(ctx, ISB_ERR_ARG, "isb_philox_bip_fluct: bad argument");
    ISB_CUDA(ctx, cudaSetDevice(ctx->device));
    double *d;
    const size_t bytes = (size_t)nr * nsteps * nunits * sizeof(double);
    ISB_TRY(isb::dev_reserve(ctx, isb::SCR_OUT, bytes, (void **)&d));
    ISB_TRY(isb::philox_bip_fluct_device(ctx, rule, seed, step_offset, layer, nunits, r0, nr, nsteps, d));
    ISB_TRY(d2h(ctx, out, d, bytes, nullptr));
    ISB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return ISB_OK;
}


// ------------------------------------------------------------------ row-sharded symmetric SCA (config 5)
static int shard_model_common(isb_ctx *ctx, int n, int n_blocks, int block, const double *Wrows, const double *h_blk,
                              const double *b_blk, uint64_t seed, double q, int prec, double wmax, isb_model **out, const char *who) {
    if (!ctx) return ISB_ERR_ARG;
    ISB_LOCK(ctx);
    if (!out) return fail(ctx, ISB_ERR_ARG, "%s: out is NULL", who);
    *out = nullptr;
    if (n <= 0 || n_blocks <= 0 || block < 0 || block >= n_blocks || n % n_blocks != 0)
        return fail(ctx, ISB_ERR_SIZE, "%s: n = %d must split evenly into %d blocks (block %d)", who, n, n_blocks, block);
    const int nb = n / n_blocks;
    const bool i8 = prec == ISB_PREC_I8X3 || prec == ISB_PREC_I8X2 || prec == ISB_PREC_I8X4;
    if (nb % (i8 ? 128 : 64) != 0)
        return fail(ctx, ISB_ERR_UNSUPPORTED, "%s: block size %d must be a multiple of %d", who, nb, i8 ? 128 : 64);
    if (prec != ISB_PREC_BF16X3 && prec != ISB_PREC_BF16X2 && prec != ISB_PREC_BF16X1 && !i8)
        return fail(ctx, ISB_ERR_ARG, "%s: prec must be ISB_PREC_BF16X3, _BF16X2, _BF16X1, _I8X3, _I8X2 or _I8X4", who);
    if (!std::isfinite(q)) return fail(ctx, ISB_ERR_NONFINITE, "%s: q is not finite", who);
    if (Wrows && !all_finite(Wrows, (size_t)nb * n)) return fail(ctx, ISB_ERR_NONFINITE, "%s: W is not finite", who);
    ISB_CUDA(ctx, cudaSetDevice(ctx->device));
    isb_model *m = new isb_model();
    m->ctx = ctx;
    ctx->refs.fetch_add(1);
    m->kind = ISB_KIND_SHARD;
    m->prec = prec;
    m->nv = m->nh = n;
    m->shard_nb = nb;
    m->shard_G = n_blocks;
    m->shard_g = block;
    std::vector<double> hn((size_t)nb, 0.0), bn((size_t)nb, 0.0);
    if (h_blk) std::copy(h_blk, h_blk + nb, hn.begin());
    if (b_blk) std::copy(b_blk, b_blk + nb, bn.begin());
    int rc = ISB_OK;
    if (cudaMalloc(&m->hb64, nb * sizeof(double)) != cudaSuccess || cudaMalloc(&m->bb64, nb * sizeof(double)) != cudaSuccess)
        rc = fail(ctx, ISB_ERR_CUDA, "%s: cudaMalloc failed", who);
    if (!rc) {
        cudaMemcpy(m->hb64, hn.data(), nb * sizeof(double), cudaMemcpyHostToDevice);
        cudaMemcpy(m->bb64, bn.data(), nb * sizeof(double), cudaMemcpyHostToDevice);
        rc = isb::shard_model_init(m, Wrows, seed, q, wmax);
    }
    if (rc) {
        isb_model_destroy(m);
        return rc;
    }
    *out = m;
    return ISB_OK;
}

int isb_shard_model_rows(isb_ctx *ctx, int n, int n_blocks, int block, const double *Wrows, const double *h_blk,
                         const double *b_blk, int prec, isb_model **out) {
    if (ctx && !Wrows) return fail(ctx, ISB_ERR_ARG, "isb_shard_model_rows: W rows are NULL");
    return shard_model_common(ctx, n, n_blocks, block, Wrows, h_blk, b_blk, 0, 0.0, prec, 0.0, out, "isb_shard_model_rows");
}

int isb_shard_model_rows_q(isb_ctx *ctx, int n, int n_blocks, int block, const double *Wrows, const double *h_blk,
                           const double *b_blk, int prec, double wmax, isb_model **out) {
    if (ctx && !Wrows) return fail(ctx, ISB_ERR_ARG, "isb_shard_model_rows_q: W rows are NULL");
    return shard_model_common(ctx, n, n_blocks, block, Wrows, h_blk, b_blk, 0, 0.0, prec, wmax, out, "isb_shard_model_rows_q");
}

int isb_shard_model_sk(isb_ctx *ctx, int n, int n_blocks, int block, uint64_t seed, double q, int prec, isb_model **out) {
    return shard_model_common(ctx, n, n_blocks, block, nullptr, nullptr, nullptr, seed, q, prec, 0.0, out, "isb_shard_model_sk");
}

int isb_sk_rows(isb_ctx *ctx, int n, uint64_t seed, int row0, int nrows, double *out) {
    if (!ctx) return ISB_ERR_ARG;
    ISB_LOCK(ctx);
    if (!out || n <= 0 || row0 < 0 || nrows < 0 || row0 + nrows > n) return fail(ctx, ISB_ERR_ARG, "isb_sk_rows: bad argument");
    ISB_CUDA(ctx, cudaSetDevice(ctx->device));
    double *d;
    const size_t bytes = (size_t)nrows * n * sizeof(double);
    ISB_TRY(isb::dev_reserve(ctx, isb::SCR_OUT, bytes, (void **)&d));
    ISB_TRY(isb::sk_rows_device(ctx, n, seed, row0, nrows, d));
    ISB_TRY(d2h(ctx, out, d, bytes, nullptr));
    ISB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return ISB_OK;
}

int isb_shard_halfstep_dev(isb_model *m, int R, int replica_offset, int layer, int rule, const void *in_full_bf16,
                           void *out_block_bf16, uint64_t seed, uint64_t step_abs, double T) {
    return isb_shard_halfstep_fused_dev(m, R, replica_offset, layer, rule, in_full_bf16, out_block_bf16, 0, nullptr, seed,
                                        step_abs, T);
}

int isb_shard_halfstep_fused_dev(isb_model *m, int R, int replica_offset, int layer, int rule, const void *in_full_bf16,
                                 void *out_block_bf16, int n_peers, void *const *peer_blocks_bf16, uint64_t seed,
                                 uint64_t step_abs, double T) {
    if (!m) return ISB_ERR_ARG;
    isb_ctx *ctx = m->ctx;
    ISB_LOCK(ctx);
    const char *who = "isb_shard_halfstep_dev";
    if (m->kind != ISB_KIND_SHARD) return fail(ctx, ISB_ERR_STATE, "%s: not a row-sharded model", who);
    if (!in_full_bf16 || !out_block_bf16 || R <= 0 || replica_offset < 0 || (layer != 0 && layer != 1) || n_peers < 0 ||
        n_peers > 7 || (n_peers > 0 && !peer_blocks_bf16) || (rule != ISB_BIP_SCA && rule != ISB_BIP_MA) || !std::isfinite(T))
        return fail(ctx, ISB_ERR_ARG, "%s: bad argument", who);
    for (int q = 0; q < n_peers; ++q)
        if (!peer_blocks_bf16[q]) return fail(ctx, ISB_ERR_ARG, "%s: NULL peer pointer", who);
    ISB_CUDA(ctx, cudaSetDevice(ctx->device));
    return isb::shard_halfstep_device(m, R, replica_offset, layer, rule, in_full_bf16, out_block_bf16, n_peers,
                                      peer_blocks_bf16, seed, step_abs, T);
}

// ------------------------------------------------------------------ instrumentation
int isb_ens_last_stats(const isb_ens *e, double *kernel_ms, int64_t *launches, int64_t *h2d_bytes, int64_t *d2h_bytes) {
    if (!e) return ISB_ERR_ARG;
    if (kernel_ms) *kernel_ms = e->last_ms;
    if (launches) *launches = e->last_launches;
    if (h2d_bytes) *h2d_bytes = e->last_h2d;
    if (d2h_bytes) *d2h_bytes = e->last_d2h;
    return ISB_OK;
}
int64_t isb_ens_last_flips(const isb_ens *e) { return e ? e->last_flips : 0; }
int64_t isb_ens_last_near_ties(const isb_ens *e) { return e ? e->last_near_ties : 0; }
int64_t isb_ens_last_exact_fallbacks(const isb_ens *e) { return e ? e->last_exact_fallbacks : 0; }
int isb_ens_set_temperature_scale(isb_ens *e, const double *scale) {
    if (!e) return ISB_ERR_ARG;
    isb_ctx *ctx = e->model->ctx;
    ISB_LOCK(ctx);
    ISB_CUDA(ctx, cudaSetDevice(ctx->device));
    if (!scale) {
        ISB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        cudaFree(e->d_tscale);
        e->d_tscale = nullptr;
        return ISB_OK;
    }
    if (!all_finite(scale, (size_t)e->R)) return fail(ctx, ISB_ERR_NONFINITE, "isb_ens_set_temperature_scale: non-finite factor");
    if (!e->d_tscale) ISB_CUDA(ctx, cudaMalloc(&e->d_tscale, (size_t)e->R * sizeof(double)));
    ISB_CUDA(ctx, cudaMemcpyAsync(e->d_tscale, scale, (size_t)e->R * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    ISB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return ISB_OK;
}
int isb_ens_set_tie_eps(isb_ens *e, double eps) {
    if (!e) return ISB_ERR_ARG;
    if (!(eps >= 0.0)) return fail(e->model->ctx, ISB_ERR_ARG, "isb_ens_set_tie_eps: eps must be >= 0");
    e->tie_eps = eps;
    return ISB_OK;
}

}  // extern "C"
