/*
 * ising_b200.h — C ABI of libising_b200.so, the B200 (sm_100a) implementation of the spin-update hot
 * path of Wandao123/IsingModel.jl.
 *
 * The reference has no FFI of its own: its boundary for this path is the Julia method set
 *   SingleSpinFlip.update!(ua, node, fluct)            src/SingleSpinFlip.jl:31,46,65
 *   OnBipartiteGraph.update!(ua, Fv, Fh)               src/OnBipartiteGraph.jl:30,53
 *   SamplingHelper.makeSampler!(ua, n; ...) step loops src/SamplingHelper.jl:28-51,110-133
 *   calcEnergy / calcLocalMagneticField / calcLocalAuxiliaryBias   src/SpinSystems.jl:68-83,139-157
 * Each entry point below names the reference lines it replaces; the Julia `ccall` stubs that bind
 * them are in isingmodel.jl_b200/julia/IsingModelB200.jl and INTEGRATION.md.
 *
 * Conventions
 *   - plain C: pointers + sizes, opaque handles, int return code (0 = ISB_OK), never throws;
 *   - every pointer argument is a HOST pointer owned by the caller for the duration of the call,
 *     except in the *_dev entry points, which take device pointers on the handle's device;
 *   - matrices are column-major with a leading dimension (Julia layout);
 *   - site / unit indices are 0-based (the Julia shim subtracts 1);
 *   - spins cross the boundary as int8 (+1 / -1), replica-major: replica r occupies
 *     s[r*ld .. r*ld + N), i.e. a Julia Matrix{Int8}(N, R);
 *   - an "ensemble" is R independent chains (replicas) of one model (the reference has one chain
 *     per SpinSystem, src/SpinSystems.jl:14-17; R = 1 reproduces it);
 *   - there is NO CPU fallback: every call needs a CUDA device and fails with ISB_ERR_CUDA otherwise.
 */
#ifndef ISING_B200_H
#define ISING_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ISB_VERSION 100 /* 0.1.0 */

typedef struct isb_ctx isb_ctx;     /* one CUDA device + error slot            */
typedef struct isb_model isb_model; /* immutable couplings resident in HBM     */
typedef struct isb_ens isb_ens;     /* R replicas of spins (+ cached fields)   */

/* return codes */
enum {
    ISB_OK = 0,
    ISB_ERR_ARG = 1,      /* NULL pointer, bad enum, negative count                       */
    ISB_ERR_SIZE = 2,     /* dimension mismatch (mirrors the error() calls of SpinSystems.jl:23,41,102-114) */
    ISB_ERR_NONFINITE = 3,/* NaN / Inf in J, h, W, T or a fluctuation                      */
    ISB_ERR_CUDA = 4,     /* CUDA runtime / driver failure, or no device                   */
    ISB_ERR_UNSUPPORTED = 5, /* shape outside what the kernels are built for               */
    ISB_ERR_NCCL = 6,
    ISB_ERR_STATE = 7     /* call not valid for this kind of model / ensemble              */
};

/* single-spin rules — src/SingleSpinFlip.jl:12-17 (Hopfield), :38-44 (Glauber == heat bath), :57-63 (Metropolis) */
enum { ISB_RULE_HOPFIELD = 0, ISB_RULE_GLAUBER = 1, ISB_RULE_METROPOLIS = 2 };
/* bipartite rules — src/OnBipartiteGraph.jl:10-16 (SCA), :45-51 (MomentumAnnealing) */
enum { ISB_BIP_SCA = 0, ISB_BIP_MA = 1 };
/* site order of a single-spin run */
enum {
    ISB_ORDER_SEQUENTIAL = 0, /* node = (start + k) mod N                                        */
    ISB_ORDER_LIST = 1,       /* node = nodes[k]   (SamplingHelper.jl:39 pre-drawn list)         */
    ISB_ORDER_RANDOM = 2,     /* node drawn by the library's Philox stream, shared by replicas    */
    ISB_ORDER_CHECKERBOARD = 3 /* periodic L x L lattices only: position k of a sweep (start = first position) visits the
                                * k-th site with (x + y) even in ascending site index, then the sites with (x + y) odd —
                                * the site list a caller of the 3-argument update! would pass for a two-colour sweep; the
                                * sites of one colour do not interact, the library updates 32 of them at once */
};
/* how an externally supplied fluctuation array is indexed */
enum {
    ISB_FLUCT_PHILOX = 0,     /* no array: library draws u by Philox4x32-10 and transforms it    */
    ISB_FLUCT_SHARED = 1,     /* one stream for all replicas                                      */
    ISB_FLUCT_PER_REPLICA = 2 /* replica r has its own stream                                     */
};
/* arithmetic of the field accumulators / storage of the couplings */
enum {
    ISB_PREC_F64 = 0, /* J and fields in double: bit-exact with the Float64 reference whenever
                         every partial sum is exactly representable (integer / dyadic J), and
                         equal up to decisions closer to zero than ~1e-13 otherwise             */
    ISB_PREC_F32 = 1, /* J and fields in float; decisions still taken in double                 */
    ISB_PREC_AUTO = 2,/* the library's choice for the model kind (dense / sparse J: F64 throughout)   */
    ISB_PREC_BF16X3 = 3, /* bipartite tensor path: W split into 3 bf16 terms, fp32 accumulation */
    ISB_PREC_BF16X1 = 4, /* bipartite tensor path: W rounded to one bf16 term (exact when W is)  */
    ISB_PREC_BF16X2 = 5, /* bipartite tensor path: 2 bf16 terms (16 mantissa bits: the split error, 2^-17
                            relative per coupling, is of the order of the fp32 accumulation error itself) */
    ISB_PREC_FP16X2 = 6, /* bipartite tensor path: 2 fp16 terms of the power-of-two pre-scaled W (11 + 11 bits + the
                            sign of the second term: 2^-24 of max|W| per coupling, i.e. W as good as rounded to
                            float) — the accuracy of _BF16X3 up to the fp32 accumulation, in two passes instead of
                            three.  Not for row-sharded models.                                                   */
    ISB_PREC_FP16X1 = 7, /* one fp16 term (2^-12 of max|W|; exact when the scaled W is fp16-representable)          */
    ISB_PREC_I8X3 = 8,   /* bipartite tensor path, INT8 DIGIT PLANES: W is rounded once to a 24-bit fixed-point grid
                            (quantum = a power of two, 2^-23 of the largest coupling; a square model's dominant diagonal —
                            the pinning term of the MultiSpinFlip embedding — is kept apart, exactly, on the same grid)
                            and contracted with tcgen05.mma.kind::i8 into int32 accumulators: the contraction itself is
                            EXACT at any depth K, so with caller-supplied fluctuations the trajectories are bit-identical
                            to the Float64 reference run on the grid couplings (isb_model_effective_couplings).  Three
                            int8 passes cost 1.5 bf16 passes.  Also valid for row-sharded models.                        */
    ISB_PREC_I8X2 = 9,   /* the same with a 16-bit grid (two planes: one bf16 pass equivalent)                             */
    ISB_PREC_I8X4 = 10   /* the same with a 32-bit grid (four planes: two bf16 pass equivalents)                           */
};

/* ------------------------------------------------------------------ context */
int isb_version(void);
int isb_device_count(void);
int isb_create(int device, isb_ctx **out);
void isb_destroy(isb_ctx *ctx);
/* Last error text of this context (never NULL); isb_last_error(NULL) = last creation error. */
const char *isb_last_error(const isb_ctx *ctx);
/* Use an existing stream (a cudaStream_t passed as void*) for all ensembles created afterwards. */
int isb_set_stream(isb_ctx *ctx, void *cuda_stream);
int isb_synchronize(isb_ctx *ctx);

/* ------------------------------------------------------------------ models */
/* SpinSystem(s, J, h): src/SpinSystems.jl:19-51.  J is n x n column-major (leading dimension ld).
 * As the reference does, a non-symmetric J is symmetrised from its upper triangle (:31-34) and the
 * diagonal is zeroed (:35-38); *warn (may be NULL) receives bit 0 / bit 1 when that happened. */
int isb_model_dense(isb_ctx *ctx, int n, const double *J, int64_t ld, const double *h, int prec,
                    int *warn, isb_model **out);
/* SpinSystem(s, J::SparseMatrixCSC, h) — the reference's tests and demo pass sparse couplings
 * (test/runtests.jl:20, demo.jl:60-62).  J in 0-based CSC (Julia's colptr .- 1, rowval .- 1, nzval); same
 * symmetrise-by-upper-triangle / zero-diagonal handling and `warn` bits as isb_model_dense.  Couplings and
 * fields are Float64; a flip touches only the stored neighbours. */
int isb_model_sparse(isb_ctx *ctx, int n, const int64_t *colptr, const int32_t *rowval, const double *nzval,
                     const double *h, int *warn, isb_model **out);
/* SpinSystemOnBipartiteGraph(sigma, tau, W, h, b): src/SpinSystems.jl:97-118. W is nv x nh. */
int isb_model_bipartite(isb_ctx *ctx, int nv, int nh, const double *W, int64_t ld,
                        const double *h, const double *b, int prec, isb_model **out);
void isb_model_destroy(isb_model *m);
/* One more owner of the model (each owner calls isb_model_destroy once): lets a host object that is copied
 * (`deepcopy(ss)`, test/runtests.jl:22-24,30-31) share the immutable device couplings with its copy. */
int isb_model_retain(isb_model *m);
/* The couplings exactly as the kernels of this model use them: W itself for ISB_PREC_F64, the sum of the stored
 * bf16 / fp16 terms or int8 digit planes (plus the split diagonal) for the tensor path.  W is nv x nh column-major with
 * leading dimension ld, like the constructor's argument.  What parity tests hand to the Float64 reference
 * (src/OnBipartiteGraph.jl:30-43) when they compare trajectories of a reduced-storage model. */
int isb_model_effective_couplings(isb_model *m, double *W, int64_t ld);
int isb_model_num_visible(const isb_model *m);
int isb_model_num_hidden(const isb_model *m); /* 0 for a general-graph model */

/* ------------------------------------------------------------------ ensembles */
int isb_ens_create(isb_model *m, int R, isb_ens **out);
void isb_ens_destroy(isb_ens *e);
int isb_ens_replicas(const isb_ens *e);
/* An independent copy of the ensemble on the same model (spins, hidden layer, per-replica temperature factors; all
 * copied device to device): what `deepcopy(ss)` of the host object maps to (test/runtests.jl:22-24,30-31). */
int isb_ens_clone(isb_ens *src, isb_ens **out);
/* Replica r takes the state of replica src[r] (src: R entries in [0, R), repeats allowed).  The spins, the cached Float64 /
 * float local fields and the fixed-point fields (whichever are valid) move with it, bit for bit.  A chain copied into slot
 * r therefore continues from exactly the state it had.  Per-replica temperature factors and flip counters belong to the
 * slot and do not move.  General-graph ensembles only (ISB_ERR_STATE for bipartite ones).  A src entry outside [0, R) is
 * ISB_ERR_ARG and leaves the ensemble unchanged. */
int isb_ens_select_replicas(isb_ens *e, const int32_t *src);
/* spinConfiguration get/set: src/SpinSystems.jl:61-62,128-129 */
int isb_ens_set_spins(isb_ens *e, const int8_t *s, int64_t ld);
int isb_ens_get_spins(isb_ens *e, int8_t *s, int64_t ld);
/* hiddenLayer get/set: src/SpinSystems.jl:130-131 */
int isb_ens_set_hidden(isb_ens *e, const int8_t *t, int64_t ld);
int isb_ens_get_hidden(isb_ens *e, int8_t *t, int64_t ld);
/* calcEnergy: src/SpinSystems.jl:68-73 / :139-145; E has R entries. */
int isb_ens_energy(isb_ens *e, double *E);
/* sum of the (visible) spins of each replica; M has R entries. */
int isb_ens_magnetization(isb_ens *e, double *M);
/* calcLocalMagneticField(ss): src/SpinSystems.jl:75-78 / :147-150; F is [R][ld], ld >= N(v). */
int isb_ens_local_field(isb_ens *e, double *F, int64_t ld);
/* calcLocalAuxiliaryBias: src/SpinSystems.jl:154-157; A is [R][ld], ld >= Nh. */
int isb_ens_local_aux_bias(isb_ens *e, double *A, int64_t ld);

/* ------------------------------------------------------------------ single-spin-flip runs */
/*
 * The step loop of makeSampler!(::SingleSpinUpdatingAlgorithm, n) (src/SamplingHelper.jl:45-49)
 * with the accept/flip rules of src/SingleSpinFlip.jl:31-36,46-55,65-74, for all R replicas:
 *   for k in 0..nsteps-1:  T <- Tsched[k / steps_per_T];  update!(ua, node_k, fluct_k)
 *
 *   order/nodes/start : see ISB_ORDER_*; nodes has nsteps entries (0-based) for ISB_ORDER_LIST.
 *   fluct_mode/fluct  : ISB_FLUCT_SHARED: fluct[nsteps]; ISB_FLUCT_PER_REPLICA: fluct[R][nsteps];
 *                       ISB_FLUCT_PHILOX: fluct ignored, (seed, step_offset) select the stream and
 *                       fluct_k = log(u/(1-u)) (Glauber), -log(u) (Metropolis), unused (Hopfield).
 *   Tsched            : nT temperatures, entry k / steps_per_T is used at step k (nT*steps_per_T >= nsteps).
 *   trace_every       : if > 0, energies and magnetisations of every replica are recorded after
 *                       each trace_every-th step into out_E / out_M ([nsteps/trace_every][R], either may be NULL).
 *   out_flips         : R entries (or NULL): number of steps that changed the spin.
 */
int isb_ssf_run(isb_ens *e, int rule, int64_t nsteps, int order, const int32_t *nodes, int start,
                int fluct_mode, const double *fluct, uint64_t seed, uint64_t step_offset,
                const double *Tsched, int64_t nT, int64_t steps_per_T, int64_t trace_every,
                double *out_E, double *out_M, int64_t *out_flips);

/* isb_ssf_run that also records the spin configuration of every replica at each trace point
 * (out_S: [nsteps/trace_every][R][ldS] int8, ldS >= N): the strided snapshots behind the streaming sampler —
 * makeSampler!'s Channel yields the state after every step (src/SamplingHelper.jl:44,48), and the host layer
 * replays it from these snapshots instead of synchronising with the device once per spin. */
int isb_ssf_run_snap(isb_ens *e, int rule, int64_t nsteps, int order, const int32_t *nodes, int start,
                     int fluct_mode, const double *fluct, uint64_t seed, uint64_t step_offset,
                     const double *Tsched, int64_t nT, int64_t steps_per_T, int64_t trace_every,
                     double *out_E, double *out_M, int64_t *out_flips, int8_t *out_S, int64_t ldS);

/* isb_ssf_run that histograms the visited configurations on the device instead of returning them: the demo's
 * "frequency of each spin configuration" plot (demo.jl:159-168: every state the sampler yields is mapped to the
 * integer whose binary digits are (1 - s_i)/2, site 1 the most significant).  hist has 2^N entries (N <= 24) and
 * is ACCUMULATED into (the caller zeroes it): every replica's configuration at every trace point adds one count. */
int isb_ssf_run_hist(isb_ens *e, int rule, int64_t nsteps, int order, const int32_t *nodes, int start,
                     int fluct_mode, const double *fluct, uint64_t seed, uint64_t step_offset,
                     const double *Tsched, int64_t nT, int64_t steps_per_T, int64_t trace_every,
                     int64_t *hist);

/* Parallel tempering (replica exchange) with the round loop on the device: R = ladders * n_levels replicas, replica
 * r = ladder * n_levels + slot; level_of[r] (in/out, a permutation of 0..n_levels-1 within each ladder) is the index into
 * levels[] that replica r holds.  Round k (absolute round K = round_offset + k) is exactly
 *   isb_ssf_run(rule, steps_per_round, order, (start + k*steps_per_round) mod N, ISB_FLUCT_PHILOX, seed,
 *               step_offset + k*steps_per_round, Tsched = {1.0}, steps_per_T = trace_every = steps_per_round)
 * with per-replica factors levels[level_of[r]], followed by one exchange in every ladder g: for
 * lo = K&1, K&1 + 2, ... <= n_levels-2, with a, b the replicas holding lo and lo+1,
 *   d = (1/levels[lo] - 1/levels[lo+1]) * (E_a - E_b)      (IEEE round-to-nearest, no contraction)
 *   u = (w + 1/2) 2^-32, w = word .x of Philox4x32-10(counter (lo32(K), hi32(K), g, 5 << 28 | lo), key seed)
 * and levels lo, lo+1 (and their temperature factors) swap between a and b when d >= 0 or u < exp(d); the spins stay.
 * E is the energy the sweep kernel traced at the last step of the round (isb_ssf_run's out_E).
 *   rule              : ISB_RULE_GLAUBER or ISB_RULE_METROPOLIS; order: sequential, random or checkerboard.
 *   out_E, out_M      : [rounds][n_levels][ladders]: energy / magnetisation traced in round k by the replica that held
 *                       level l during that round (before the swaps).
 *   out_Q             : [rounds][n_levels][ladders/2]: overlap (sum_i s_i^a s_i^b) / N of the replicas of ladders 2p and
 *                       2p+1 that held level l during round k, at its end (an even number of ladders is required).
 *   out_accepted      : [n_levels-1] accepted swaps per level pair in this call (proposed: ladders x rounds of the
 *                       pair's parity).  out_flips: [R] flips per replica summed over the rounds.
 * Every output may be NULL.  On return level_of holds the final assignment and the ensemble's temperature factors are
 * levels[level_of], so a later isb_ssf_run continues the ladders; two calls of K rounds (start, step_offset and
 * round_offset continued) equal one call of 2K rounds bit for bit.  rounds = 0 is a no-op. */
int isb_ssf_run_pt(isb_ens *e, int rule, int n_levels, const double *levels, int64_t rounds, int64_t steps_per_round,
                   int order, int start, uint64_t seed, uint64_t step_offset, uint64_t round_offset,
                   int32_t *level_of, double *out_E, double *out_M, double *out_Q,
                   int64_t *out_accepted, int64_t *out_flips);

/* Population annealing: R = n_pop * P replicas, population p = slots p*P .. p*P + P - 1 (P <= 2^20).  Temperature step k
 * (absolute index K = T_offset + k) is exactly
 *   isb_ssf_run(rule, steps_per_T, order, (start + k*steps_per_T) mod N, ISB_FLUCT_PHILOX, seed,
 *               step_offset + k*steps_per_T, Tsched = {T[k]}, steps_per_T = trace_every = steps_per_T)
 * followed, when k < nT - 1 or T_next > 0, by one resampling of every population towards T' = T[k+1] (or T_next):
 *   db = 1/T' - 1/T[k];  a_r = -db * E_r;  x_r = exp(a_r - max_r a_r)      (IEEE round-to-nearest, no contraction)
 *   W_r = floor(x_r * 2^32) (uint64),  C_r = W_0 + ... + W_r,  S = C_{P-1}        (exact integers)
 *   U   = word .x of Philox4x32-10(counter (lo32(K), hi32(K), p, 6 << 28), key seed)
 *   slot j of the population takes the state (isb_ens_select_replicas) of the smallest r with
 *   C_r > floor((j * 2^32 + U) * S / (P * 2^32))                                (128-bit integer arithmetic)
 *   lnQ[k][p] = max_r a_r + ln(sum_r x_r / P);  family[j] <- family[parent(j)]
 * (r, j: indices within the population).  E_r is the energy the sweep kernel traced at the last step (isb_ssf_run's out_E).
 *   rule: Glauber or Metropolis; order: sequential, random or checkerboard (lattices); T[k] > 0 and finite; T_next = 0: none.
 *   out_E, out_M [nT][R] by slot (before that step's resampling); out_lnQ [nT - 1 + (T_next > 0)][n_pop];
 *   family [R] in/out (any int32 labels, may be NULL); out_flips [R] per slot over the call.
 * Every output may be NULL.  Two calls (T[0..a) with T_next = T[a], then T[a..b); start, step_offset and T_offset
 * continued) equal one call of T[0..b) bit for bit.  Per-replica temperature factors must be unset (ISB_ERR_STATE).
 * nT = 0 is a no-op. */
int isb_ssf_run_pa(isb_ens *e, int rule, int n_pop, int64_t nT, const double *T, double T_next, int64_t steps_per_T,
                   int order, int start, uint64_t seed, uint64_t step_offset, uint64_t T_offset, int32_t *family,
                   double *out_E, double *out_M, double *out_lnQ, int64_t *out_flips);

/* Swendsen-Wang cluster sweeps of an ensemble of a SPARSE model (isb_model_sparse: any graph, periodic lattices included;
 * n <= 16384 sites, ISB_ERR_UNSUPPORTED above; dense and bipartite ensembles: ISB_ERR_STATE).  Energy convention as
 * everywhere: E = -sum_{i<j} J_ij s_i s_j - sum_i h_i s_i.  Sweep k of the call (absolute index K = sweep_offset + k) of
 * replica r runs at T_r(k) = Tsched[k / sweeps_per_T] * scale[r] (the isb_ens_set_temperature_scale factors, 1 when unset),
 * the product isb_ssf_run forms:
 *   bonds     the pairs (i, j), i < j, J_ij != 0 after the constructor's symmetrisation, numbered e = 0, 1, ... in order
 *             of i, then j (row i of the stored CSR, columns > i).  Bond e is active when J_ij s_i s_j > 0 and
 *             u(w_e) < 1 - exp(-2|J_ij| / T_r(k)), w_e = word e & 3 of Philox4x32-10(counter (lo32 K, hi32 K, r,
 *             7 << 28 | e >> 2), key seed), u(w) = (w + 1/2) 2^-32; exp in double, IEEE round-to-nearest, no contraction;
 *   clusters  the connected components of the active bonds; the ROOT of a cluster is its smallest site;
 *   fields    on a grid, so that the cluster sums are exact and independent of order: e_h = the smallest integer with
 *             max|h| <= 2^e_h, q = 2^(e_h - 30), hq_i = rint(h_i / q) (every hq_i = 0 when h = 0).  The chain samples the
 *             Boltzmann distribution of the fields q hq, which differ from h by at most 2^-31 max|h| each;
 *   flips     for cluster C with root rho: S_C = sum_{i in C} hq_i s_i (exact int64), x = 2 q S_C / T_r(k),
 *             P = 1 / (1 + exp(x)); every spin of C flips when u(z) < P, z = word rho & 3 of Philox4x32-10(counter
 *             (lo32 K, hi32 K, r, 8 << 28 | rho >> 2), key seed).  P = 1/2 exactly when h = 0.  This is the heat-bath
 *             choice of each cluster's orientation given its bonds: detailed balance holds with fields and with couplings
 *             of either sign.
 * The device's double exp and a replay's may differ by an ulp: a decision can differ only when u falls between the two,
 * with probability of order 2^-53 per decision.
 *   out_E, out_M   [nsweeps / trace_every][R]: energy (in double, exact for dyadic J and h; its summation order differs from
 *                  isb_ens_energy) and magnetisation after the flips of every trace_every-th sweep;
 *   out_csq        same shape: sum over that sweep's clusters of |C|^2, the improved estimator of the susceptibility
 *                  (chi = <sum |C|^2> / N at h = 0);
 *   out_flips      [R]: spins flipped during the call.
 * Every output may be NULL.  ISB_ERR_ARG: nsweeps < 0, sweeps_per_T < 1, trace_every < 0 or, when nsweeps > 0, no schedule
 * (nT < 1), a schedule shorter than nsweeps (nT * sweeps_per_T < nsweeps) or a temperature T_r(k) <= 0 the call would use;
 * ISB_ERR_NONFINITE: a non-finite one.  An error leaves the ensemble unchanged; nsweeps = 0 is a no-op.  The result is
 * bit-identical from run to run and does not depend on the launch configuration; two calls (sweep_offset and schedule
 * continued) equal one call.  The cached fields of the single-spin kernels are rebuilt by the next isb_ssf_run. */
int isb_sw_run(isb_ens *e, int64_t nsweeps, uint64_t seed, uint64_t sweep_offset, const double *Tsched, int64_t nT,
               int64_t sweeps_per_T, int64_t trace_every, double *out_E, double *out_M, int64_t *out_csq,
               int64_t *out_flips);

/* Fluctuations exactly as ISB_FLUCT_PHILOX generates them inside isb_ssf_run, for parity tests:
 * out[r*nsteps + k], r in [r0, r0+nr). rule selects the transform. prec as the model's. */
int isb_philox_fluct(isb_ctx *ctx, int rule, int prec, uint64_t seed, uint64_t step_offset,
                     int r0, int nr, int64_t nsteps, double *out);
/* Site list exactly as ISB_ORDER_RANDOM generates it. */
int isb_philox_nodes(isb_ctx *ctx, int n, uint64_t seed, uint64_t step_offset, int64_t nsteps,
                     int32_t *out);
/* Raw Philox4x32-10 blocks (for known-answer tests): out[4*i..] = philox(ctr[4*i..], key). */
int isb_philox_raw(isb_ctx *ctx, const uint32_t *ctr, const uint32_t key[2], int nblocks,
                   uint32_t *out);

/* ------------------------------------------------------------------ bipartite (block Gibbs) runs */
/*
 * The step loop of makeSampler!(::UpdatingAlgorithmOnBipartiteGraph, n) (src/SamplingHelper.jl:127-131)
 * with update! of src/OnBipartiteGraph.jl:30-43 (SCA) / :53-66 (MomentumAnnealing):
 *   hidden <- sgn+(2(W' sigma + b) - Fh*T [.* hidden]);  visible <- sgn+(2(W hidden + h) - Fv*T [.* visible])
 *
 *   fluct_mode SHARED: Fv[nsteps][nv], Fh[nsteps][nh]; PER_REPLICA: Fv[R][nsteps][nv], Fh[R][nsteps][nh];
 *   PHILOX: drawn inside the kernel (logistic for SCA, exponential for MA).
 *   out_E: [nsteps/trace_every][R] energies (may be NULL).
 */
int isb_bip_run(isb_ens *e, int rule, int64_t nsteps, int fluct_mode, const double *Fv,
                const double *Fh, uint64_t seed, uint64_t step_offset, const double *Tsched,
                int64_t nT, int64_t steps_per_T, int64_t trace_every, double *out_E);

/* isb_bip_run that also records both layers of every chain at each trace point (out_Sv: [ntr][R][ldSv],
 * out_Sh: [ntr][R][ldSh] int8; either may be NULL): the snapshots behind the streaming sampler of
 * makeSampler!(::UpdatingAlgorithmOnBipartiteGraph, n) (src/SamplingHelper.jl:124-132). */
int isb_bip_run_snap(isb_ens *e, int rule, int64_t nsteps, int fluct_mode, const double *Fv, const double *Fh,
                     uint64_t seed, uint64_t step_offset, const double *Tsched, int64_t nT, int64_t steps_per_T,
                     int64_t trace_every, double *out_E, int8_t *out_Sv, int64_t ldSv, int8_t *out_Sh,
                     int64_t ldSh);

/* Fluctuations as ISB_FLUCT_PHILOX draws them in isb_bip_run: layer 0 = visible, 1 = hidden;
 * out[(r - r0)][k][unit]. */
int isb_philox_bip_fluct(isb_ctx *ctx, int rule, int prec, uint64_t seed, uint64_t step_offset,
                         int layer, int nunits, int r0, int nr, int64_t nsteps, double *out);


/* ------------------------------------------------------------------ row-sharded synchronous SCA (one process per GPU) */
/*
 * The large dense-J case (BASELINE config 5): the MultiSpinFlip SCA of an N-spin model, i.e. the bipartite SCA
 * (src/OnBipartiteGraph.jl:30-43) on the embedding W = (J + qI)/2, h/2, h/2, sigma = tau = s (demo.jl:82-90),
 * with W too large for one GPU.  Rank `block` of `n_blocks` owns the output units
 * [block*nb, (block+1)*nb), nb = n / n_blocks, of BOTH half-steps (W is symmetric) and holds only W[block rows, :].
 * The spin matrices live in CALLER-OWNED device buffers (the caller allocates them and gathers the sampled blocks
 * of every rank between half-steps; isb_shard_run_* below does both):
 *   full layer  : bf16 [n_blocks][R][nb]   (block-major, +1/-1)        — the K operand of a half-step
 *   own block   : bf16 [R][nb], one buffer per layer                    — what this rank samples (on entry it
 *                 holds the block's previous values, which MomentumAnnealing multiplies into the noise)
 * (ISB_PREC_I8X* models: the same buffers hold int8 +1/-1 instead of bf16 — half the bytes to all-gather.)
 * Noise is the library's Philox stream indexed by GLOBAL (replica, step, unit), so the trajectory does not
 * depend on the number of blocks.
 */
/* W rows given by the caller: Wrows is [nb][n] row-major (rows block*nb .. of the symmetric W). */
int isb_shard_model_rows(isb_ctx *ctx, int n, int n_blocks, int block, const double *Wrows, const double *h_blk,
                         const double *b_blk, int prec, isb_model **out);
/* The same for the int8 digit-plane formats, whose fixed-point grid must be identical on every rank: wmax = the
 * largest off-diagonal |W| of the WHOLE matrix (<= 0: use this block's own maximum). */
int isb_shard_model_rows_q(isb_ctx *ctx, int n, int n_blocks, int block, const double *Wrows, const double *h_blk,
                           const double *b_blk, int prec, double wmax, isb_model **out);
/* Synthetic SK instance generated on the device, never materialised in full: J_ij = J_ji ~ N(0, 1/n) from the
 * counter RNG (seed), W = (J + qI)/2, zero fields. */
int isb_shard_model_sk(isb_ctx *ctx, int n, int n_blocks, int block, uint64_t seed, double q, int prec,
                       isb_model **out);
/* Rows row0 .. row0+nrows of that synthetic J (out is [nrows][n] row-major), for parity tests. */
int isb_sk_rows(isb_ctx *ctx, int n, uint64_t seed, int row0, int nrows, double *out);
int isb_model_shard_block(const isb_model *m); /* nb, 0 for other models */
/* One half-step of this rank's block (layer 1: hidden from the full visible layer, 0: visible from the full
 * hidden layer): own <- sgn+(2 (W[block,:] . in + bias) - F T [.* own]) for all R replicas.  All pointers are
 * DEVICE pointers on the context's device; the kernel is enqueued on the context's stream (isb_set_stream). */
/* R replicas whose global indices start at replica_offset (isb_shard_run_* splits the replicas into two groups and
 * hides one group's exchange under the other group's GEMM: chains are independent). */
int isb_shard_halfstep_dev(isb_model *m, int R, int replica_offset, int layer, int rule,
                           const void *in_full, void *out_block, uint64_t seed, uint64_t step_abs, double T);

/* The step loop of the row-sharded SCA inside the library (no torch, no Python on the path): one run object per rank
 * owns the gathered spin matrices and this rank's blocks, splits the replicas into two groups and hides one group's
 * exchange under the other group's contraction.  The exchange after every half-step is the path's one collective
 * (BASELINE config 5: "all-gather of the spin vector each synchronous step"):
 *   ISB_EXCH_LOCAL  one block, no exchange;
 *   ISB_EXCH_NCCL   ncclAllGather on a side stream.  libnccl.so.2 is resolved with dlopen at first use; give the run the
 *                   caller's communicator (isb_shard_run_set_nccl_comm: an ncclComm_t of n_blocks ranks, this rank =
 *                   block) or let it create one: rank 0 calls isb_nccl_unique_id, sends the 128 bytes to every rank by
 *                   its own means (MPI, a file, torch.distributed), every rank calls isb_shard_run_init_nccl;
 *   ISB_EXCH_COPY   copy-engine pushes into the peers' gathered matrices + flag words (CUDA IPC; one process per GPU on
 *                   one box): every rank exports a 64-byte handle (isb_shard_run_ipc_export), the caller passes them
 *                   around, every rank imports every other rank's (isb_shard_run_ipc_import).
 * The trajectory depends neither on the number of blocks nor on the exchange (noise indexed by global replica, step,
 * unit): parity tests compare with the unsharded tensor path. */
typedef struct isb_shard_run isb_shard_run;
enum { ISB_EXCH_LOCAL = 0, ISB_EXCH_NCCL = 1, ISB_EXCH_COPY = 2 };
int isb_shard_run_create(isb_model *shard_model, int R, int exchange, isb_shard_run **out);
void isb_shard_run_destroy(isb_shard_run *s);
int isb_nccl_unique_id(void *id128);
int isb_shard_run_init_nccl(isb_shard_run *s, const void *id128);
int isb_shard_run_set_nccl_comm(isb_shard_run *s, void *nccl_comm);
int isb_shard_run_ipc_export(isb_shard_run *s, void *handle64);
int isb_shard_run_ipc_import(isb_shard_run *s, int rank, const void *handle64);
/* Cross-rank barrier of the copy-engine exchange (every rank calls it; returns when all have). */
int isb_shard_run_barrier(isb_shard_run *s);
/* S: [R][ld] int8 +-1, the same on every rank; both layers start from it (sigma = tau = s, demo.jl:82-90).  Collective
 * for ISB_EXCH_COPY (ends with the barrier). */
int isb_shard_run_set_spins(isb_shard_run *s, const int8_t *S, int64_t ld);
/* layer 0: the spin configuration (visible copy), 1: the hidden copy; identical on every rank. */
int isb_shard_run_get_spins(isb_shard_run *s, int layer, int8_t *S, int64_t ld);
/* nsteps synchronous steps of rule ISB_BIP_SCA / _MA (src/OnBipartiteGraph.jl:30-43,53-66); step k runs at
 * Tsched[min(k, nT - 1)] and draws the noise of global step step_offset + k.  Collective: every rank calls it with the
 * same arguments. */
int isb_shard_run_steps(isb_shard_run *s, int rule, int64_t nsteps, const double *Tsched, int64_t nT, uint64_t seed,
                        uint64_t step_offset);
/* Device time (ms) and kernel launches of the last isb_shard_run_steps call, and the number of replica groups. */
int isb_shard_run_last_stats(const isb_shard_run *s, double *device_ms, int64_t *launches, int *n_groups);

/* ------------------------------------------------------------------ instrumentation */
/* Device time (ms, CUDA events on the ensemble's stream) of the kernels of the last *_run call,
 * number of kernel launches it made, and bytes copied host->device / device->host by it. */
int isb_ens_last_stats(const isb_ens *e, double *kernel_ms, int64_t *launches, int64_t *h2d_bytes,
                       int64_t *d2h_bytes);
/* Sum over replicas of accepted flips in the last isb_ssf_run (for the roofline's rows-fetched count). */
int64_t isb_ens_last_flips(const isb_ens *e);
/* Decisions of the last run whose |2h - fT| was below tie_eps (near-tie audit, SURVEY 7.2). */
int64_t isb_ens_last_near_ties(const isb_ens *e);
/* Decisions of the last run that the fixed-point sweep kernels could not settle from their integer fields and took on
 * the reference's fresh Float64 row dot instead (DESIGN §3; 0 for runs on the Float64 kernels). */
int64_t isb_ens_last_exact_fallbacks(const isb_ens *e);
int isb_ens_set_tie_eps(isb_ens *e, double eps);
/* Per-replica temperature factors (scale: R entries, NULL clears them): replica r runs every later *_run call at
 * T_r(k) = Tsched[k] * scale[r].  R reference objects that differ only in their `temperature` field
 * (src/SingleSpinFlip.jl:40,59; src/OnBipartiteGraph.jl:12,47) are one ensemble: temperature scans, parallel
 * tempering (swap = permute the factors, the spins stay where they are). */
int isb_ens_set_temperature_scale(isb_ens *e, const double *scale);

#ifdef __cplusplus
}
#endif
#endif /* ISING_B200_H */
