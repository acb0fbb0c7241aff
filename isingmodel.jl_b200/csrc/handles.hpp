// handles.hpp — host-side objects behind the opaque handles of include/ising_b200.h.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <mutex>
#include <string>

#include "../../include/ising_b200.h"

struct isb_devbuf {
    void *p = nullptr;
    size_t cap = 0;
};

struct isb_ctx {
    std::atomic<int> refs{1};    // the creator + every live model: destroyed when the last one lets go
    int device = 0;
    int num_sms = 148;
    size_t smem_optin = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    isb_devbuf scratch[18];      // grow-only device staging buffers (see isb::dev_reserve)
    // Every entry point that uses the stream, the events or the scratch buffers holds this lock for its whole
    // (synchronous) duration: calls on one context are serialised, different contexts run concurrently.
    std::recursive_mutex mtx;
};

// a run that starts this many sweeps (or more) after the last fresh field computation recomputes the cached fields
#define ISB_FIELD_REFRESH_SWEEPS 64

enum { ISB_KIND_DENSE = 0, ISB_KIND_BIPARTITE = 1, ISB_KIND_SHARD = 2, ISB_KIND_SPARSE = 3 };

struct isb_model {
    std::atomic<int> refs{1};    // the creator + every live ensemble
    isb_ctx *ctx = nullptr;
    int kind = ISB_KIND_DENSE;
    int prec = ISB_PREC_F64;
    // ---- dense: N sites, padded to Npad = 32*NPL (NPL a power of two) for the sweep kernel
    int n = 0, npad = 0, npl = 0;
    bool fast_ok = false;        // N <= 1024: register-resident sweep kernel applies
    bool j_is_f32 = false;       // storage type of the permuted copy used by the sweep kernel
    double *J64 = nullptr;       // natural layout [npad][npad] (row i contiguous; symmetric)
    void *Jperm = nullptr;       // permuted columns (isb::ssf_perm_pos), double or float, [npad][npad]
    double *h64 = nullptr;       // [npad]
    // near-tie guard of the single-spin kernels: 0 when every coupling and field is a small dyadic number (all sums are
    // exact), else 2^-30 of the largest row sum of |J| + |h| (see SsfParams::guard)
    double guard = 0.0;
    // fixed-point copy for the sweep kernels (N <= 1024, Float64 models; DESIGN §3): Jint = round(J / fix_q), permuted like
    // Jperm with VEC = 4, fix_q = 2^-k with every row sum of |Jint| below 2^30; fix_margin = M >= max_i (e_i + dot
    // rounding) / fix_q, e_i = sum_j |J_ij - fix_q Jint_ij| (0 when every coupling is a multiple of fix_q)
    bool fixed_ok = false;
    int32_t *Jfix = nullptr;
    double fix_q = 1.0;
    int fix_margin = 0;
    // ---- bipartite: nv visible, nh hidden
    int nv = 0, nh = 0;
    double *W64 = nullptr;       // [nv][nh]  (row i = visible unit i; contiguous over hidden)
    double *Wt64 = nullptr;      // [nh][nv]
    double *hb64 = nullptr;      // visible bias [nv]
    double *bb64 = nullptr;      // hidden bias  [nh]
    // tensor-core operands (bf16 split terms, K-major, padded) — filled by bip_tc.cu when prec is BF16X*
    void *tc = nullptr;
    // ---- row-sharded symmetric SCA (kind SHARD): this rank owns units [shard_g*shard_nb, (shard_g+1)*shard_nb)
    int shard_nb = 0, shard_G = 0, shard_g = 0;
    // ---- sparse general-graph model (kind SPARSE): CSR rows of the symmetric J, owned by sparse.cu
    void *sp = nullptr;
};

struct isb_ens {
    isb_model *model = nullptr;
    int R = 0;
    int8_t *spins = nullptr;     // [R][npad]   (dense)  or  [R][nvpad] (bipartite visible)
    int8_t *hidden = nullptr;    // [R][nhpad]
    int64_t lds = 0, ldh = 0;    // row strides of the two arrays (bytes == elements)
    void *fields = nullptr;      // cached local fields [R][npad], double or float
    int fields_rule_sign = 0;    // 0 = invalid, +1 = J s + h (Glauber/Metropolis), -1 = J s - h (Hopfield)
    // The cached fields are maintained incrementally (+-2 J[i,:] per accepted flip); for couplings whose sums round, the
    // incremental value drifts from a fresh row dot by a few ulp per flip.  A run that starts after this many steps
    // since the last fresh computation recomputes them first (sequential row dots, the reference's order).
    int64_t steps_since_refresh = 0;
    int32_t *ifields = nullptr;  // fixed-point fields [R][npad] (exact integers Jint s; allocated by the first fixed-point run)
    bool ifields_ok = false;     // false: rebuilt from the spins by the next fixed-point run
    // second set of the state buffers for isb_ens_select_replicas (gather into them, then swap the pointers); each is
    // allocated by the first selection that moves it
    int8_t *spins2 = nullptr;
    void *fields2 = nullptr;
    int32_t *ifields2 = nullptr;
    unsigned long long *d_flips = nullptr;   // [R]
    unsigned long long *d_counters = nullptr; // [0] near ties, [1] exact fallbacks of the fixed-point kernels
    double tie_eps = 0.0;
    double *d_tscale = nullptr;  // optional per-replica temperature factors [R]: T_r(k) = Tsched[k] * tscale[r]
    // last-run statistics
    double last_ms = 0.0;
    int64_t last_launches = 0, last_h2d = 0, last_d2h = 0, last_flips = 0, last_near_ties = 0, last_exact_fallbacks = 0;
    void *tc = nullptr;          // tensor-core path state (bf16 spin matrices), owned by bip_tc.cu
};

namespace isb {

int fail(isb_ctx *ctx, int code, const char *fmt, ...);
// The permuted column layout of the sweep kernel's couplings (isb_model::Jperm, and Jfix with VEC = 4): site k*32 + lane
// of a row sits at position (k / VEC)*32*VEC + lane*VEC + k % VEC, so that a lane loads the couplings of its sites k .. k +
// VEC - 1 with one vector load (VEC = min(16 bytes / coupling size, NPL); ssf_kernel's apply_row).
__host__ __device__ constexpr int ssf_perm_pos(int site, int vec) {
    const int k = site >> 5, lane = site & 31;
    return (k / vec) * (32 * vec) + lane * vec + k % vec;
}
__host__ __device__ constexpr int ssf_perm_site(int pos, int vec) {   // the inverse of ssf_perm_pos
    const int kv = pos / (32 * vec), rm = pos % (32 * vec);
    return (kv * vec + rm % vec) * 32 + rm / vec;
}
// Near-tie guard of a general-graph model from its couplings (n values per row at vals[i * ld + j], or a flat list with
// rows given by rowptr) and fields: see isb_model::guard.
double ssf_guard_from(const double *absrowsum, const double *vals, size_t nvals, const double *h, int n);
// Grow-only device scratch buffer `slot` of the context, at least `bytes` long.
int dev_reserve(isb_ctx *ctx, int slot, size_t bytes, void **out);
enum { SCR_NODES = 0, SCR_FLUCT = 1, SCR_T = 2, SCR_E = 3, SCR_M = 4, SCR_FLUCT2 = 5, SCR_OUT = 6, SCR_TMP = 7,
       SCR_TC0 = 8, SCR_TC1 = 9, SCR_S = 10, SCR_S2 = 11, SCR_HIST = 12, SCR_PT_STATE = 13, SCR_PT_E = 14, SCR_PT_M = 15,
       SCR_PT_Q = 16, SCR_PA_STATE = 17 };

#define ISB_LOCK(ctx) std::lock_guard<std::recursive_mutex> isb_lock_guard_((ctx)->mtx)

#define ISB_CUDA(ctx, call)                                                                      \
    do {                                                                                         \
        cudaError_t _e = (call);                                                                 \
        if (_e != cudaSuccess)                                                                   \
            return isb::fail((ctx), ISB_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), \
                             __FILE__, __LINE__);                                                \
    } while (0)

// ssf.cu
// The sweeps of every single-spin entry point (isb_ssf_run*, and each round / temperature step of isb_ssf_run_pt /
// isb_ssf_run_pa), on arguments the entry point has checked: for ISB_ORDER_RANDOM the Philox site list into d_nodes
// [nsteps] first, then dense models up to 1024 sites on the register-resident kernel, everything else on the
// neighbour-list kernel (which hands periodic lattices to the lattice kernels).
int ssf_sweep_device(isb_ens *e, int rule, int64_t nsteps, int order, int32_t *d_nodes, int start, int fluct_mode,
                     const double *d_fluct, uint64_t seed, uint64_t step_offset, const double *d_T, int64_t steps_per_T,
                     int64_t trace_every, double *d_E, double *d_M, int8_t *d_S);
int ssf_ensure_fields(isb_ens *e, int sign);
size_t ssf_field_elem_size(const isb_model *m);
int philox_fluct_device(isb_ctx *ctx, int rule, uint64_t seed, uint64_t step_offset, int r0, int nr,
                        int64_t nsteps, double *d_out);
int philox_nodes_device(isb_ctx *ctx, int n, uint64_t seed, uint64_t step_offset, int64_t nsteps,
                        int32_t *d_out);
int philox_raw_device(isb_ctx *ctx, const uint32_t *d_ctr, uint32_t k0, uint32_t k1, int nblocks,
                      uint32_t *d_out);
int dense_energy_device(isb_ens *e, double *d_E);
int dense_field_device(isb_ens *e, double *d_F, int64_t ld);  // natural J s + h in double
int magnetization_device(isb_ens *e, double *d_M);
// counts[index(config)] += 1 for each of the `count` configurations in d_S ([count][n] int8), n <= 24
int config_histogram_device(isb_ctx *ctx, const int8_t *d_S, int64_t count, int n, unsigned long long *d_hist);

// sparse.cu
int sparse_model_init(isb_model *m, int n, const int64_t *colptr, const int32_t *rowval, const double *nzval, int *warn);
void sparse_model_free(isb_model *m);
bool sparse_model_lattice(const isb_model *m);   // a periodic lattice the lattice kernels run (ISB_ORDER_CHECKERBOARD)
void sparse_model_set_guard(isb_model *m, const double *h_host);  // near-tie guard from the stored couplings and h
int sparse_field_device(isb_ens *e, double *d_out, int64_t ld, int nout, double hsign);
int sparse_energy_device(isb_ens *e, double *d_E);
int ssf_sparse_run_device(isb_ens *e, int rule, int64_t nsteps, int order, const int32_t *d_nodes, int start,
                          int fluct_mode, const double *d_fluct, uint64_t seed, uint64_t step_offset, const double *d_T,
                          int64_t steps_per_T, int64_t trace_every, double *d_E, double *d_M, int8_t *d_S);

// lattice.cu (periodic square lattices recognised by sparse_model_init)
} // namespace isb
#include <utility>
#include <vector>
namespace isb {
void *lattice_detect(isb_ctx *ctx, int n, const std::vector<std::vector<std::pair<int, double>>> &rows);
void lattice_free(void *lat);
int lattice_side(const void *lat);
int ssf_lattice_run_device(isb_ens *e, void *lat, int rule, int64_t nsteps, int order, int start, int fluct_mode, const double *d_fluct,
                           uint64_t seed, uint64_t step_offset, const double *d_T, int64_t steps_per_T, int64_t trace_every,
                           double *d_E, double *d_M, int8_t *d_S);

// tempering.cu: `rounds` rounds of isb_ssf_run_pt on the context stream, no host synchronisation between rounds.  Round k
// is one sweep launch of steps_per_round steps (traced E / M of its last step into d_Eround / d_Mround [R]), the overlap
// kernel when d_recQ is given, then the exchange kernel (level_of, e->d_tscale, acceptance counts, flip totals, records).
int ssf_pt_run_device(isb_ens *e, int rule, int n_levels, const double *d_levels, int64_t rounds, int64_t steps_per_round,
                      int order, int start, uint64_t seed, uint64_t step_offset, uint64_t round_offset, int32_t *d_nodes,
                      const double *d_T, int32_t *d_level_of, double *d_Eround, double *d_Mround, double *d_recE,
                      double *d_recM, double *d_recQ, unsigned long long *d_accepted, unsigned long long *d_flips_total);

// population.cu: isb_ens_select_replicas on the context stream (d_src: R device entries, checked by the caller), and the
// temperature loop of isb_ssf_run_pa (buffers of PaDevice; db[k] = 1/T[k+1] - 1/T[k] per resampling, n_res of them).
int ens_select_device(isb_ens *e, const int32_t *d_src);
struct PaDevice {
    const double *T;                        // [nT]
    int32_t *nodes;                         // [steps_per_T] (random order)
    double *recE, *recM;                    // [nT][R] records (NULL: recE -> E [R] only, no M)
    double *E;                              // [R] energies of the step when recE is NULL
    double *a, *bmax, *bx, *pmax, *lnQ;     // [R], [n_pop*nb] x 2, [n_pop], [n_res][n_pop]
    unsigned long long *cloc, *bW, *flips_total;   // [R], [n_pop*nb], [R]
    int32_t *parent, *fam[2];               // [R]; family ping-pong (NULL: no family)
};
int ssf_pa_run_device(isb_ens *e, int rule, int n_pop, int64_t nT, const double *db, int64_t n_res, int64_t steps_per_T,
                      int order, int start, uint64_t seed, uint64_t step_offset, uint64_t T_offset, const PaDevice &d,
                      int *fam_final);

// bip_exact.cu
int bip_run_exact_device(isb_ens *e, int rule, int64_t nsteps, int fluct_mode, const double *d_Fv,
                         const double *d_Fh, uint64_t seed, uint64_t step_offset, const double *d_T,
                         int64_t steps_per_T, int64_t trace_every, double *d_E, int8_t *d_Sv, int8_t *d_Sh);
int bip_snapshot(isb_ens *e, int64_t ntr, int8_t *d_Sv, int8_t *d_Sh);
int bip_energy_device(isb_ens *e, double *d_E);
int bip_field_device(isb_ens *e, int layer, double *d_out, int64_t ld);  // layer 0: W tau + h, 1: W' sigma + b
int philox_bip_fluct_device(isb_ctx *ctx, int rule, uint64_t seed, uint64_t step_offset, int layer,
                            int nunits, int r0, int nr, int64_t nsteps, double *d_out);

// bip_tc.cu (tcgen05 path)
int bip_tc_model_init(isb_model *m, const double *W_host_rowmajor_vh);
void bip_tc_model_free(isb_model *m);
int bip_tc_ens_init(isb_ens *e);
void bip_tc_ens_free(isb_ens *e);
int shard_model_init(isb_model *m, const double *Wrows /*[nb][n] or NULL*/, uint64_t seed, double q, double wmax);
int bip_tc_effective_couplings(isb_model *m, double *W_host_rowmajor_vh);
int shard_halfstep_device(isb_model *m, int R, int replica_offset, int layer, int rule, const void *in_full, void *out_block,
                          int n_peers, void *const *peer_blocks, uint64_t seed, uint64_t step_abs, double T);
int shard_elem_size(const isb_model *m);  // bytes per +-1 of the spin matrices of a row-sharded model (1 int8, 2 bf16)
int sk_rows_device(isb_ctx *ctx, int n, uint64_t seed, int row0, int nrows, double *d_out);
int bip_run_tc_device(isb_ens *e, int rule, int64_t nsteps, int fluct_mode, const double *d_Fv,
                      const double *d_Fh, uint64_t seed, uint64_t step_offset, const double *d_T,
                      int64_t steps_per_T, int64_t trace_every, double *d_E, int8_t *d_Sv, int8_t *d_Sh);

}  // namespace isb
