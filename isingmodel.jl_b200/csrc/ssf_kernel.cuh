// ssf_kernel.cuh — K1: replica-batched single-spin-flip sweeps (Hopfield / Glauber / Metropolis).
//
// Replaces, for R chains at once, the reference's per-step path
//   SamplingHelper.makeSampler! loop            src/SamplingHelper.jl:45-49
//     -> SingleSpinFlip.update!(ua, node, f)    src/SingleSpinFlip.jl:31-36,46-55,65-74
//        -> calcLocalMagneticField(ua, i)       src/SpinSystems.jl:80-83   (an O(N) row dot per step)
//
// Design (B200-first, not a translation):
//   * one warp per chain; the chain's N local fields live in registers (site i <-> lane i%32,
//     register i/32), its spins in one 32-bit mask per lane;
//   * the local field is maintained incrementally: an accepted flip of site i adds +-2*J[i,:] to the
//     fields (J symmetric, src/SpinSystems.jl:31-38), so a row of J is touched only on accepted flips;
//   * every chain of a CTA visits the sites in the same order, so one copy of row i serves all of
//     them: a producer warp streams the rows of J through a shared-memory ring with 1-D bulk async
//     copies (TMA, cp.async.bulk -> UBLKCP) completing on mbarriers, G rows per ring slot;
//   * sequential sweeps are processed 32 sites at a time *speculatively*: all 32 lanes evaluate the
//     decision of their own site at once; a ballot finds the first lane that flips, its row is
//     applied, and only the lanes after it are re-evaluated.  This is exactly the sequential
//     single-site dynamics (a site's decision is taken with the fields left by all earlier sites).
//   * decisions are taken in double with the reference's operation order: 2*h, f*T, (f*T)*s, subtract,
//     compare with heaviside(0)=1 (src/SpinSystems.jl:163-171).
#pragma once
#include <stdio.h>

#include <type_traits>

#include "common.cuh"

namespace isb {

constexpr int SSF_G = 8;  // rows of J per ring slot (a power of two; 8 measured best against 2, 4 and 16: DESIGN §7)

struct SsfParams {
    const void *J;  // permuted couplings [npad][ldj] (double or float)
    int64_t ldj;    // row stride in elements
    const double *hext;  // external field [npad]
    int8_t *spins;       // [R][lds]
    int64_t lds;
    void *fields;  // [R][npad] (HT)
    int n, npad, R;
    int rule;
    double ecoef;  // energy = -1/2 sum s*fld - ecoef * sum h*s
    int64_t nsteps;
    int start;
    const int32_t *nodes;
    int fluct_mode;
    const double *fluct;
    int64_t fluct_pitch;   // per-replica fluctuations: steps per replica of the whole run (= nsteps unless the run is segmented)
    uint64_t seed, step_offset;
    const double *Tsched;
    const double *tscale;  // per-replica temperature factors [R] or NULL
    int64_t steps_per_T;
    int64_t trace_every;
    double *out_E, *out_M;
    int8_t *out_S;   // spin snapshots at the trace points: [ntr][R][ldS] (or NULL)
    int64_t ldS;
    unsigned long long *flips;
    unsigned long long *near_ties;
    double tie_eps;
    int nw;  // consumer warps (chains) per CTA
    int NG;  // ring slots
    // Adaptive row delivery (TMA kernels): the run is cut into epochs of SSF_EPOCH steps.  In a *streamed* epoch
    // the producer pushes every visited row through the ring (cost: one row per step per CTA, shared by its
    // chains); in an *on-demand* epoch each chain reads the rows of its own accepted flips straight from L2
    // (cost: one row per flip per chain).  After each epoch the CTA compares its flip count with the step
    // count and streams the next epoch iff flips >= od_ratio * steps (low temperatures go on-demand).
    float od_ratio;
    PhiloxKeys keys;  // the ten Philox round keys of `seed` (read straight from the constant bank)
    // Near-tie guard (couplings whose sums round: guard > 0).  The incrementally maintained field differs from the
    // reference's fresh row dot (src/SpinSystems.jl:80-83) by a few ulp; when a decision quantity is closer to zero than
    // `guard`, the lane recomputes its field as that sequential dot (natural J64 rows, ascending j) before it decides,
    // so that exact ties and exact cancellations of the reference are reproduced.  0 (and the kernel instantiated
    // without the guard) for models whose arithmetic is exact (integer / dyadic couplings) and for couplings drawn from
    // a continuum (more than 64 distinct magnitudes: exact ties have probability zero; the near-tie audit still counts).
    double guard;
    const double *J64;  // natural layout [npad][ld64]
    int64_t ld64;
    double hsign;       // +1: J s + h, -1: J s - h (Hopfield)
    // Fixed-point instantiation (HT = JT = int32_t): p.J holds Jint = round(J / q), the cached fields are the exact
    // integers F = Jint s (no h), and every decision the thresholds of fixed_thresholds cannot settle is taken on
    // ssf_exact_field, the reference's own row dot.  fix_margin = M >= (e_max + dot rounding) / q, DESIGN §3.
    double fix_q, fix_invq;
    int fix_margin;
    unsigned long long *fallbacks;  // decisions taken on ssf_exact_field (fixed-point kernels)
};
constexpr int SSF_EPOCH = 1024;        // steps per streamed epoch
constexpr int SSF_EPOCH_OD = 8 * 1024;  // steps per on-demand epoch: chains re-synchronise 8x less often

// consumer warps (chains) per CTA for a chain that keeps `field_regs` 32-bit registers of local
// fields per lane: 15 warps -> 128 registers/thread, 21 -> 96, 29 -> 64 (one CTA per SM, +1 producer warp)
__host__ __device__ constexpr int ssf_max_chains(int field_regs) {
    return field_regs > 32 ? 14 : (field_regs > 16 ? 20 : 28);
}

template <typename HT, int NPL>
struct SsfCfg {
    // (int32 fixed-point fields are budgeted like Float64 ones: their decision step and fallback need the registers)
    static constexpr int kFieldRegs = NPL * (std::is_same<HT, int32_t>::value ? 2 : (int)sizeof(HT) / 4);
    static constexpr int kMaxChains = ssf_max_chains(kFieldRegs);
    static constexpr int kMaxThreads = 32 * (kMaxChains + 1);
};

// compile-time loop: f(integral_constant<int, I>) for I in [0, N) — keeps register-array indices static
template <int I, int N, typename F>
__device__ __forceinline__ void static_for(F &&f) {
    if constexpr (I < N) {
        f(std::integral_constant<int, I>{});
        static_for<I + 1, N>(f);
    }
}

template <typename JT, int VEC>
struct alignas(sizeof(JT) * VEC) JPack {
    JT v[VEC];
};

// hf[k] with k known only at run time and WARP-UNIFORM (k = site / 32): a switch that ptxas turns into a short
// uniform branch tree (not dynamic register indexing, which would push the fields to local memory)
template <typename HT, int NPL>
__device__ __forceinline__ HT field_sel(const HT (&hf)[NPL], int k) {
    HT v = hf[0];
#define ISB_CASE(i) \
    case i:         \
        if constexpr (i < NPL) v = hf[i < NPL ? i : 0]; \
        break;
    switch (k) {
        ISB_CASE(1) ISB_CASE(2) ISB_CASE(3) ISB_CASE(4) ISB_CASE(5) ISB_CASE(6) ISB_CASE(7) ISB_CASE(8)
        ISB_CASE(9) ISB_CASE(10) ISB_CASE(11) ISB_CASE(12) ISB_CASE(13) ISB_CASE(14) ISB_CASE(15) ISB_CASE(16)
        ISB_CASE(17) ISB_CASE(18) ISB_CASE(19) ISB_CASE(20) ISB_CASE(21) ISB_CASE(22) ISB_CASE(23) ISB_CASE(24)
        ISB_CASE(25) ISB_CASE(26) ISB_CASE(27) ISB_CASE(28) ISB_CASE(29) ISB_CASE(30) ISB_CASE(31)
        default: break;
    }
#undef ISB_CASE
    return v;
}

// hf[k] = v for a warp-uniform run-time k (the counterpart of field_sel; rare path)
template <typename HT, int NPL>
__device__ __forceinline__ void field_set(HT (&hf)[NPL], int k, HT v) {
    static_for<0, NPL>([&](auto I) {
        if (I.value == k) hf[I.value] = v;
    });
}
// The reference's fresh local field of site i: sum_j J[i][j] s_j sequentially over ascending j, then +- h_i.  The
// chain's spins are spread over the warp (site j <-> lane j % 32, bit j / 32 of sw): every lane walks the same loop,
// lanes with `want` accumulate their own row.  Rare (near ties only), deliberately not inlined.
static __device__ __noinline__ double ssf_exact_field(const double *J64, int64_t ld64, const double *hext, double hsign, int n,
                                               uint32_t sw, int i, bool want) {
    double acc = 0.0;
    const double *row = J64 + (int64_t)i * ld64;
    for (int j = 0; j < n; ++j) {
        const uint32_t w = __shfl_sync(0xffffffffu, sw, j & 31);
        if (want) {
            const double v = __ldg(row + j);
            acc = __dadd_rn(acc, ((w >> (j >> 5)) & 1u) ? v : -v);
        }
    }
    return want ? __dadd_rn(acc, hsign * __ldg(hext + i)) : 0.0;
}

// Decision thresholds of the fixed-point kernels for one site and one window (fts = the site's f*T or (f*T)*s_i, hh =
// hsign * h_i; both fixed through the window).  pred(F) is the reference's decision with the dot replaced by F * q
// (exact: F is an integer below 2^30, q a power of two); it is monotone in F, so a = min{F in [-B, B] : pred(F)} splits
// the integers.  The reference's own dot lies within M * q of F * q (DESIGN §3), hence
//   F >= a + M  ->  the reference flips up,   F < a - M  ->  it flips down,   otherwise: ask ssf_exact_field.
// With M = 0 (couplings that are exact multiples of q) lo == hi and nothing falls back.  a starts at ceil(t), t the
// real-valued boundary, and is settled by evaluating pred itself; a boundary that does not settle in 8 steps (huge |h|
// against q) sends every value to the exact path.
__device__ __forceinline__ void fixed_thresholds(double fts, double hh, double q, double invq, int M, int &lo, int &hi) {
    constexpr int B = (1 << 30) + 1;
    auto pred = [&](int F) { return !(__dsub_rn(2.0 * __dadd_rn(__dmul_rn((double)F, q), hh), fts) < 0.0); };
    const double t = ceil(__dmul_rn(__dsub_rn(0.5 * fts, hh), invq));
    int a = !(t > (double)-B) ? -B : (t > (double)B ? B : (int)t);
    int it = 0;
    while (it < 8 && a > -B && pred(a - 1)) --a, ++it;
    while (it < 8 && a < B && !pred(a)) ++a, ++it;
    if (it >= 8) {
        lo = -0x7fffffff - 1;
        hi = 0x7fffffff;
        return;
    }
    lo = a - M;   // |a| <= 2^30 + 1 and M <= 2^10 (model creation): no overflow
    hi = a + M;
}

// GUARD: the near-tie guard (SsfParams::guard) is compiled in — a separate instantiation, because its rare slow path
// costs the hot loop registers (measured: 195 -> 232 ms on the C2 schedule when it is merely present).
template <typename HT, typename JT, int NPL, bool LIST, bool TMA, bool GUARD = false>
__global__ void __launch_bounds__(SsfCfg<HT, NPL>::kMaxThreads, 1) ssf_kernel(const SsfParams p) {
    // int32 fields and couplings: the fixed-point path (sequential order, plain kernel, no traces, no tie audit; see SsfParams)
    constexpr bool FIXED = std::is_same<HT, int32_t>::value;
    static_assert(!FIXED || (std::is_same<JT, int32_t>::value && !LIST && !TMA && !GUARD), "fixed-point: plain sequential sweeps only");
    constexpr int G = SSF_G;
    constexpr int NPAD = NPL * 32;
    constexpr int ROWB = NPAD * (int)sizeof(JT);
    constexpr int VEC = (16 / (int)sizeof(JT)) < NPL ? (16 / (int)sizeof(JT)) : NPL;
    constexpr int NCH = NPL / VEC;
    constexpr uint32_t FULL = 0xffffffffu;

    extern __shared__ __align__(128) unsigned char smem_raw[];
    JT *ring = reinterpret_cast<JT *>(smem_raw);
    uint64_t *full_bar = reinterpret_cast<uint64_t *>(smem_raw + (size_t)p.NG * G * ROWB);
    uint64_t *empty_bar = full_bar + p.NG;
    uint64_t *ep_bar = empty_bar + p.NG;    // consumers -> producer: "epoch finished" (count = chains of this CTA)
    uint64_t *go_bar = ep_bar + 1;          // producer -> consumers: "mode of the next epoch decided"
    unsigned int *ep_flips = reinterpret_cast<unsigned int *>(go_bar + 1);  // flips of the CTA in the current epoch
    volatile int *ep_mode = reinterpret_cast<volatile int *>(ep_flips + 1); // 1 = streamed, 0 = on demand

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nw = p.nw;
    const int first_chain = blockIdx.x * nw;
    const int nactive = min(nw, p.R - first_chain);
    const int NG = p.NG;
    const JT *Jg = reinterpret_cast<const JT *>(p.J);

    if constexpr (TMA) {
        if (threadIdx.x == 0) {
            for (int s = 0; s < NG; ++s) {
                mbar_init(&full_bar[s], 1);
                mbar_init(&empty_bar[s], (uint32_t)(nactive > 0 ? nactive : 1));
            }
            mbar_init(ep_bar, (uint32_t)(nactive > 0 ? nactive : 1));
            mbar_init(go_bar, 1);
            *ep_flips = 0u;
            *ep_mode = 1;
            mbar_fence_init();
        }
        __syncthreads();
    }

    // ------------------------------------------------------------------ producer warp
    if (warp == nw) {
        if constexpr (TMA) {
            if (lane == 0) {
                // adaptive delivery is decided per CTA
                const bool adaptive = p.od_ratio > 0.f && nactive > 0;
                int site = p.start;
                int slot = 0;
                uint32_t ph = 0;  // (slot, ph) of the next streamed group, kept incrementally (no 64-bit divisions)
                int64_t issued = 0;
                uint32_t ep = 0;
                int ep_len = SSF_EPOCH, prev_len = SSF_EPOCH;
                for (int64_t t0 = 0; t0 < p.nsteps; t0 += ep_len, ++ep) {
                    bool stream = true;
                    if (adaptive && ep > 0) {
                        mbar_wait(ep_bar, (ep - 1) & 1u);  // every chain of the CTA has finished epoch ep - 1
                        stream = (float)(*ep_flips) >= p.od_ratio * (float)prev_len;
                        *ep_flips = 0u;
                        *ep_mode = stream ? 1 : 0;
                        mbar_arrive(go_bar);
                    }
                    ep_len = stream ? SSF_EPOCH : SSF_EPOCH_OD;
                    prev_len = ep_len;
                    const int64_t esteps = p.nsteps - t0 < ep_len ? p.nsteps - t0 : ep_len;
                    if (!stream) {
                        if constexpr (!LIST) site = (int)(((int64_t)site + esteps) % p.n);
                        continue;
                    }
                    const int64_t nq = (esteps + G - 1) / G;
                    for (int64_t q = 0; q < nq; ++q, ++issued) {
                        // slot free in this CTA: its chains released the group that used it NG groups ago (a CTA
                        // without chains instead waits until that group's bytes have landed, so the barrier is
                        // never armed twice per phase)
                        if (nactive > 0)
                            mbar_wait(&empty_bar[slot], ph ^ 1u);
                        else if (issued >= NG)
                            mbar_wait(&full_bar[slot], ph ^ 1u);
                        const int64_t left = esteps - q * G;
                        const int rows = left < G ? (int)left : G;
                        mbar_arrive_expect_tx(&full_bar[slot], (uint32_t)(rows * ROWB));
                        for (int g = 0; g < rows; ++g) {
                            int i;
                            if constexpr (LIST) {
                                i = __ldg(&p.nodes[t0 + q * G + g]);
                            } else {
                                i = site;
                                if (++site == p.n) site = 0;
                            }
                            bulk_g2s(ring + ((size_t)slot * G + g) * NPAD, Jg + (int64_t)i * p.ldj, ROWB, &full_bar[slot]);
                        }
                        if (++slot == NG) {
                            slot = 0;
                            ph ^= 1u;
                        }
                    }
                }
                // no bulk copy may still be in flight when the CTA retires: wait for the last min(issued, NG) groups
                const int last = (int)(issued < NG ? issued : NG);
                for (int b = 0; b < last; ++b) {
                    if (--slot < 0) {
                        slot = NG - 1;
                        ph ^= 1u;
                    }
                    mbar_wait(&full_bar[slot], ph);
                }
            }
        }
    } else if (warp < nactive) {

    // ------------------------------------------------------------------ consumer warp = one chain
    const int r = first_chain + warp;
    HT hf[NPL];
    uint32_t sw = 0;
    {
        const HT *fr = reinterpret_cast<const HT *>(p.fields) + (int64_t)r * NPAD;
        const int8_t *sr = p.spins + (int64_t)r * p.lds;
#pragma unroll
        for (int k = 0; k < NPL; ++k) {
            hf[k] = fr[k * 32 + lane];
            sw |= (sr[k * 32 + lane] > 0 ? 1u : 0u) << k;
        }
    }
    const bool metro = p.rule == 2;
    const int rule = p.rule;
    const bool audit = p.tie_eps > 0.0;
    // T_r = Tsched * tscale[r] (x 1.0 is exact); the factor is re-read whenever a schedule entry is fetched rather than
    // kept live: two more registers in the sweep loop cost 3 % on C2
#define ISB_TSC() (p.tscale ? __ldg(&p.tscale[r]) : 1.0)
    unsigned long long nflips = 0, nties = 0, nfall = 0;
    // Ring position of this chain within the current (streamed) epoch: qcur = group of the epoch being read
    // (-1: none yet), held = it has not been released; cslot / cph walk the ring across epochs (only streamed
    // groups are ever pushed, so producer and chains stay in step).  te = steps done in the current epoch.
    int qcur = -1;
    bool held = false;
    int cslot = -1;
    uint32_t cph = 0;
    bool stream = TMA;  // delivery mode of the current epoch
    int te = 0;
    int ep_len = SSF_EPOCH;  // length of the current epoch (on-demand epochs are longer)
    uint32_t ep_idx = 0;
    unsigned int ep_nflips = 0;
    const bool adaptive = TMA && p.od_ratio > 0.f;

    auto release_held = [&]() {
        if (held) {
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty_bar[cslot]);
            held = false;
        }
    };
    // make group q of this epoch the held one: release the previous groups in order, wait for each new one
    auto advance_to = [&](int q) {
        if constexpr (TMA) {
            while (qcur < q) {
                release_held();
                ++qcur;
                if (++cslot == NG) {
                    cslot = 0;
                    cph ^= 1u;
                }
                mbar_wait(&full_bar[cslot], cph);
                held = true;
            }
        }
    };
    // called when te == ep_len (t = global step count): finish the epoch, learn the next one's delivery mode
    auto epoch_boundary = [&](int64_t t) {
        if constexpr (TMA) {
            if (stream) {
                advance_to((SSF_EPOCH - 1) / G);  // consume (and then release) every group of the epoch
                release_held();
            }
            qcur = -1;
            nflips += ep_nflips;
            if (adaptive && t < p.nsteps) {
                __syncwarp();
                if (lane == 0) {
                    atomicAdd(ep_flips, ep_nflips);
                    mbar_arrive(ep_bar);
                }
                mbar_wait(go_bar, ep_idx & 1u);
                stream = *ep_mode != 0;
            }
            ep_len = stream ? SSF_EPOCH : SSF_EPOCH_OD;
            ep_nflips = 0;
            ++ep_idx;
            te = 0;
        }
    };
    // fields += d * J[row], in batches of at most 8 vector loads (32 registers in flight): the compiler barrier
    // keeps it from hoisting all NCH loads above the FMAs, which would spill the register-resident fields
    auto apply_row = [&](const JT *row, HT d) {
        constexpr int BATCH = NCH < 8 ? NCH : 8;
#pragma unroll
        for (int c0 = 0; c0 < NCH; c0 += BATCH) {
            JPack<JT, VEC> pk[BATCH];
#pragma unroll
            for (int c = 0; c < BATCH; ++c)
                pk[c] = *reinterpret_cast<const JPack<JT, VEC> *>(row + (c0 + c) * 32 * VEC + lane * VEC);
#pragma unroll
            for (int c = 0; c < BATCH; ++c)
#pragma unroll
                for (int b = 0; b < VEC; ++b) hf[(c0 + c) * VEC + b] += d * (HT)pk[c].v[b];
            asm volatile("" ::: "memory");
        }
    };
    auto write_trace = [&](int64_t idx) {
        double sf = 0.0, sh = 0.0;
        int m = 0;
#pragma unroll
        for (int k = 0; k < NPL; ++k) {
            const int site = k * 32 + lane;
            const bool up = (sw >> k) & 1u;
            const double f = (double)hf[k];
            sf += up ? f : -f;
            if (site < p.n) {
                const double hv = __ldg(&p.hext[site]);
                sh += up ? hv : -hv;
                m += up ? 1 : -1;
            }
        }
        sf = warp_sum(sf);
        sh = warp_sum(sh);
        m = warp_sum_int(m);
        if (lane == 0) {
            if (p.out_E) p.out_E[idx * p.R + r] = -0.5 * sf - p.ecoef * sh;
            if (p.out_M) p.out_M[idx * p.R + r] = (double)m;
        }
        if (p.out_S) {
            int8_t *so = p.out_S + (idx * p.R + r) * p.ldS;
#pragma unroll
            for (int k = 0; k < NPL; ++k)
                if (k * 32 + lane < p.n) so[k * 32 + lane] = ((sw >> k) & 1u) ? (int8_t)1 : (int8_t)-1;
        }
    };

    const uint64_t spT = (uint64_t)p.steps_per_T;
    int64_t next_trace = p.trace_every > 0 ? p.trace_every : INT64_MAX;
    int64_t trace_idx = 0;
    int64_t cached_ti = -1;
    double cachedT = 0.0;

    if constexpr (!LIST) {
        // ---------------------------------------------------------- sequential order, 32-site speculation
        int64_t t = 0;
        int site = p.start;
        uint64_t ti = 0, tr = 0;  // t = ti*spT + tr
        while (t < p.nsteps) {
            const int k = site >> 5;
            const int l_first = site & 31;
            int len = 32 - l_first;
            if (p.n - site < len) len = p.n - site;
            if (p.nsteps - t < len) len = (int)(p.nsteps - t);
            if (next_trace - t < len) len = (int)(next_trace - t);
            if (TMA && ep_len - te < len) len = ep_len - te;
            const int off = lane - l_first;
            const bool mine = off >= 0 && off < len;
            // temperature of my step
            double Tl;
            {
                const uint64_t a_hi = tr + (uint64_t)(len - 1);
                if (a_hi < spT) {
                    if ((int64_t)ti != cached_ti) {
                        cachedT = __dmul_rn(__ldg(&p.Tsched[ti]), ISB_TSC());  // scaled once per schedule entry
                        cached_ti = (int64_t)ti;
                    }
                    Tl = cachedT;
                } else {
                    const uint64_t a = tr + (uint64_t)(mine ? off : 0);
                    Tl = __dmul_rn(__ldg(&p.Tsched[ti + a / spT]), ISB_TSC());
                }
            }
            // fluctuation of my step
            double f = 0.0;
            if (rule != 0 && mine) {
                const int64_t tl = t + off;
                if (p.fluct_mode == 0) {
                    f = ssf_fluct_from_word(
                        rule, philox_step_word_k(p.keys, DOM_SSF_FLUCT, (uint32_t)r, p.step_offset + (uint64_t)tl));
                } else if (p.fluct_mode == 1) {
                    f = __ldg(&p.fluct[tl]);
                } else {
                    f = __ldg(&p.fluct[(int64_t)r * p.fluct_pitch + tl]);
                }
            }
            const double ftl = __dmul_rn(f, Tl);
            bool mybit = (sw >> k) & 1u;
            // hk mirrors hf[k] (my own site's field) for this block; both receive identical updates
            HT hk = field_sel<HT, NPL>(hf, k);
            const int kpos = (k / VEC) * (32 * VEC) + lane * VEC + (k % VEC);
            uint32_t rem = __ballot_sync(FULL, mine);
            [[maybe_unused]] int flo = 0, fhi = 0;
            if constexpr (FIXED) {
                const double fts = metro ? (mybit ? ftl : -ftl) : ftl;
                fixed_thresholds(fts, p.hsign * __ldg(&p.hext[k * 32 + lane]), p.fix_q, p.fix_invq, p.fix_margin, flo, fhi);
            }
            while (true) {
                bool nb;
                uint32_t fm;   // lanes still to decide whose decision flips their spin
                if constexpr (FIXED) {
                    nb = hk >= fhi;
                    const bool near = !nb && hk >= flo && ((rem >> lane) & 1u);
                    const uint32_t nm = __ballot_sync(FULL, near);
                    if (nm) {   // rare: decide on the reference's fresh sequential row dot
                        const double ex = ssf_exact_field(p.J64, p.ld64, p.hext, p.hsign, p.n, sw, k * 32 + lane, near);
                        const double fts = metro ? (mybit ? ftl : -ftl) : ftl;
                        if (near) nb = !(__dsub_rn(2.0 * ex, fts) < 0.0);
                        nfall += __popc(nm);
                    }
                    fm = __ballot_sync(FULL, nb != mybit) & rem;
                } else {
                double h2 = 2.0 * (double)hk;
                const double fts = metro ? (mybit ? ftl : -ftl) : ftl;
                double x = __dsub_rn(h2, fts);
                if constexpr (GUARD) {
                    const bool near = fabs(x) < p.guard && ((rem >> lane) & 1u);
                    if (__any_sync(FULL, near)) {   // rare: decide on the reference's fresh sequential row dot
                        const double ex = ssf_exact_field(p.J64, p.ld64, p.hext, p.hsign, p.n, sw, k * 32 + lane, near);
                        if (near) {
                            hk = (HT)ex;
                            h2 = 2.0 * (double)hk;
                            x = __dsub_rn(h2, fts);
                        }
                        field_set<HT, NPL>(hf, k, hk);
                    }
                }
                nb = !(x < 0.0);  // heaviside(0) = 1, src/SpinSystems.jl:163-171
                fm = __ballot_sync(FULL, nb != mybit) & rem;
                if (audit) {
                    const uint32_t tm = __ballot_sync(FULL, fabs(x) < p.tie_eps) & rem;
                    nties += __popc(fm ? (tm & ((2u << (__ffs(fm) - 1)) - 1u)) : tm);
                }
                }
                if (fm == 0) break;
                const int l0 = __ffs(fm) - 1;
                const uint32_t upto = (2u << l0) - 1u;  // lanes <= l0 (l0 == 31 -> all ones)
                const bool up = (__ballot_sync(FULL, nb) >> l0) & 1u;
                const HT d = up ? (HT)2 : (HT)-2;
                // one update path over a generic pointer (ring slot or L2): two specialised copies (LDS / LDG)
                // made ptxas hoist 16 x LDG.128 above the FMAs and spill the register-resident fields
                const JT *row;
                if (TMA && stream) {
                    const int se = te + (l0 - l_first);  // step within the epoch
                    advance_to(se / G);
                    row = ring + ((size_t)cslot * G + (size_t)(se & (G - 1))) * NPAD;
                } else {
                    row = Jg + (int64_t)(k * 32 + l0) * p.ldj;
                }
                hk += d * (HT)row[kpos];
                apply_row(row, d);
                if (lane == l0) {
                    sw ^= 1u << k;
                    mybit = !mybit;
                }
                ++ep_nflips;
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
            te += len;
            if (TMA && stream) advance_to((te - 1) / G);
            if (t == next_trace) {
                write_trace(trace_idx++);
                next_trace += p.trace_every;
            }
            if (TMA && te == ep_len) epoch_boundary(t);
        }
    } else {
        // ---------------------------------------------------------- explicit site list, one step at a time
        uint64_t ti = 0, tr = 0;
        double Tcur = 0.0;
        int node_batch = 0;
        double f_batch = 0.0;
        for (int64_t t = 0; t < p.nsteps; ++t) {
            const int j = (int)(t & 31);
            if (j == 0) {  // every 32 steps: each lane fetches the node and fluctuation of step t + lane
                const int64_t tl = t + lane;
                node_batch = 0;
                f_batch = 0.0;
                if (tl < p.nsteps) {
                    node_batch = __ldg(&p.nodes[tl]);
                    if (rule != 0) {
                        if (p.fluct_mode == 0) {
                            f_batch = ssf_fluct_from_word(rule, philox_step_word_k(p.keys, DOM_SSF_FLUCT, (uint32_t)r,
                                                                                  p.step_offset + (uint64_t)tl));
                        } else if (p.fluct_mode == 1) {
                            f_batch = __ldg(&p.fluct[tl]);
                        } else {
                            f_batch = __ldg(&p.fluct[(int64_t)r * p.fluct_pitch + tl]);
                        }
                    }
                }
            }
            if ((int64_t)ti != cached_ti) {
                Tcur = __dmul_rn(__ldg(&p.Tsched[ti]), ISB_TSC());
                cached_ti = (int64_t)ti;
            }
            const int site = __shfl_sync(FULL, node_batch, j);
            const double f = __shfl_sync(FULL, f_batch, j);
            const int k = site >> 5, l = site & 31;
            const double ft = __dmul_rn(f, Tcur);
            const bool mybit = (sw >> k) & 1u;
            double h2 = 2.0 * (double)field_sel<HT, NPL>(hf, k);
            const double fts = metro ? (mybit ? ft : -ft) : ft;
            double x = __dsub_rn(h2, fts);
            if constexpr (GUARD) {
                const bool near = lane == l && fabs(x) < p.guard;
                if (__any_sync(FULL, near)) {
                    const double ex = ssf_exact_field(p.J64, p.ld64, p.hext, p.hsign, p.n, sw, site, near);
                    if (near) {
                        field_set<HT, NPL>(hf, k, (HT)ex);
                        h2 = 2.0 * (double)(HT)ex;
                        x = __dsub_rn(h2, fts);
                    }
                }
            }
            const bool nb = !(x < 0.0);
            uint32_t code = (nb != mybit ? 1u : 0u) | (nb ? 2u : 0u) | (fabs(x) < p.tie_eps ? 4u : 0u);
            code = __shfl_sync(FULL, code, l);
            if (audit) nties += (code >> 2) & 1u;
            if (TMA && stream) advance_to(te / G);
            if (code & 1u) {
                const HT d = (code & 2u) ? (HT)2 : (HT)-2;
                apply_row((TMA && stream) ? ring + ((size_t)cslot * G + (size_t)(te & (G - 1))) * NPAD
                                          : Jg + (int64_t)site * p.ldj,
                          d);
                if (lane == l) sw ^= 1u << k;
                ++ep_nflips;
            }
            ++te;
            if (++tr == spT) {
                tr = 0;
                ++ti;
            }
            if (t + 1 == next_trace) {
                write_trace(trace_idx++);
                next_trace += p.trace_every;
            }
            if (TMA && te == ep_len) epoch_boundary(t + 1);
        }
    }

    // ------------------------------------------------------------------ write the chain back
    {
        HT *fr = reinterpret_cast<HT *>(p.fields) + (int64_t)r * NPAD;
        int8_t *sr = p.spins + (int64_t)r * p.lds;
#pragma unroll
        for (int k = 0; k < NPL; ++k) {
            fr[k * 32 + lane] = hf[k];
            if (k * 32 + lane < p.n) sr[k * 32 + lane] = ((sw >> k) & 1u) ? (int8_t)1 : (int8_t)-1;
        }
        if (lane == 0) {
            p.flips[r] = nflips + ep_nflips;
            if (nties) atomicAdd(p.near_ties, nties);
            if (nfall) atomicAdd(p.fallbacks, nfall);
        }
    }
    }  // consumer warp
}

}  // namespace isb
