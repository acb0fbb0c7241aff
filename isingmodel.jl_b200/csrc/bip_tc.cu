// bip_tc.cu — K3/K4: block-Gibbs half-steps as tcgen05 GEMMs with the sampling rule fused into the epilogue.
//
// Replaces, for R chains at once (ISB_PREC_BF16X3 / ISB_PREC_BF16X1 bipartite models),
//   hidden  <- sgn+(2 (W' sigma + b) - Fh T [.* hidden])     src/OnBipartiteGraph.jl:35-38 (SCA), :58-61 (MA)
//   visible <- sgn+(2 (W tau + h)   - Fv T [.* visible])     src/OnBipartiteGraph.jl:39-42 (SCA), :62-65 (MA)
//   with W' sigma + b = calcLocalAuxiliaryBias, W tau + h = calcLocalMagneticField (src/SpinSystems.jl:147-157).
//
// One half-step is D[replica, unit] = S_in[replica, :] . Wop[unit, :] (a dense contraction over the input layer):
//   A operand  = the spin matrix S_in [R][K] in bf16 (+-1 is exact), K-major, 128 replicas per tile (UMMA M = 128)
//   B operand  = the couplings Wop [units][K] in bf16, K-major, BN <= 256 units per tile (UMMA N = BN);
//                W is stored as P bf16 terms W = W1 + W2 + W3 (P = 3: 24 mantissa bits, fp32-exact split;
//                P = 1: W rounded to bf16, exact when W is bf16-representable, e.g. small integers);
//   D          = fp32 accumulators in TMEM (2 stages x 256 columns), all P terms accumulate into the same D.
// Warp-specialised persistent kernel, one CTA per SM, in CTA pairs (cta_group::2: the two CTAs of a cluster run one
// M = 256 MMA, each loading its own 128 replicas of A and half of the coupling tile, so every SM pulls half of the
// coupling bytes from L2; single CTAs were measured slower on every workload, DESIGN §3):
//   warp 0 = TMA producer (cp.async.bulk.tensor, 128B swizzle, smem ring of 6 slots, mbarrier complete_tx)
//   warp 1 = MMA issuer (tcgen05.mma.kind::f16 by one elected lane of the leader CTA, tcgen05.commit frees the slot)
//   warp 2 = TMEM allocator
//   warps 4-15 = epilogue: tcgen05.ld the accumulators, draw the noise (Philox4x32-10, same words as the
//                Float64 path), apply the rule, write the new layer as bf16 (next GEMM's operand),
//                overlapping the next tile's MMAs; the canonical int8 spins are refreshed per run / trace point.
// The producer and issuer warps run their loops warp-uniformly and pick the issuing lane with elect.sync, so that
// descriptors and barrier addresses stay in uniform registers (see the note at the MMA issuer).
//
// Operand formats (template parameter FMT): 0 = bf16 terms, 1 = fp16 terms of the pre-scaled couplings, 2 = INT8 DIGIT
// PLANES (ISB_PREC_I8X*): W is rounded once to a P x 8-bit fixed-point grid (quantum q0 = 2^e, a power of two) and
// stored as P planes of balanced base-256 digits; spins are int8 +-1 (the ensemble's canonical arrays ARE the A
// operand).  The P planes of a tile of `bn` units are STACKED along the MMA's N dimension — the coupling matrix is
// stored tile-major [tile][plane][unit in tile][K], so one tcgen05.mma.kind::i8 of N = P * bn <= 256 columns contracts
// the spin tile with all planes at once (the A tile is fetched and read from shared memory once per K block, not once
// per plane) and leaves plane t EXACTLY in the int32 TMEM columns [t * bn, (t + 1) * bn) of the tile's accumulator stage;
// the epilogue recombines field = q0 * sum_t 256^(P-1-t) acc_t — no rounding anywhere in the contraction, at any K.
// One int8 pass costs half a bf16 pass (2x tensor rate, half the operand bytes), so 24-bit couplings cost 1.5 bf16-pass
// equivalents (bf16x3: 3, fp16x2: 2).  A square model's diagonal (the pinning term q/2 of the MultiSpinFlip embedding, demo.jl:82-90, 64x
// larger than the couplings) is split off and added in the epilogue from the unit's own input spin, so that the
// fixed-point grid is scaled to the off-diagonal couplings.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <stdlib.h>

#include <type_traits>
#include <utility>
#include <vector>

#include "common.cuh"
#include "handles.hpp"

namespace isb {

constexpr int TC_BM = 128;      // replicas per tile (UMMA M)
constexpr int TC_BK = 64;       // K elements per stage, 16-bit operands (128 bytes = one swizzle span)
constexpr int TC_BK8 = 128;     // K elements per stage, int8 digit planes (the same 128 bytes)
constexpr int TC_PMAX = 4;      // coupling terms / digit planes
constexpr int TC_BN_MAX = 256;  // units per tile (UMMA N), runtime BN <= 256, multiple of 16
constexpr int TC_STAGES = 6;     // smem ring slots
constexpr int TC_A_BYTES = TC_BM * TC_BK * 2;            // 16 KiB: this CTA's 128 replicas
constexpr int TC_B_BYTES = TC_BN_MAX / 2 * TC_BK * 2;    // 16 KiB: this CTA's half of the coupling tile
constexpr int TC_STAGE_BYTES = TC_A_BYTES + TC_B_BYTES;
constexpr int TC_EPI_WARPS = 12;  // a multiple of 4: equal shares of the four TMEM lane quadrants
constexpr int TC_CW = 16;         // accumulator columns (units) per epilogue chunk
static_assert(TC_EPI_WARPS % 4 == 0, "epilogue shape");
constexpr int TC_THREADS = 32 * (4 + TC_EPI_WARPS);
constexpr int TC_HALVES = TC_EPI_WARPS / 4;     // epilogue warps per TMEM lane quadrant
constexpr int TC_GW = TC_CW * TC_HALVES;        // accumulator columns the epilogue warps cover per round
constexpr int TC_SIG_MAX = 32;                  // chain-resident mode: progress barriers per layer
constexpr size_t TC_SMEM = (size_t)TC_STAGES * TC_STAGE_BYTES + 1024 /*alignment slack*/ + 1024 /*barriers*/;
static_assert((2 * TC_STAGES + 8 + 2 * TC_SIG_MAX) * 8 <= 1024, "barrier block");

struct TcModel {
    int P = 1;
    // operand format: bf16 terms (8 significant bits each), or fp16 terms (11 bits each; ISB_PREC_FP16X*): the
    // couplings are then pre-scaled by the power of two `wscale` (max |W| -> [2^13, 2^14)) so that the residual term
    // stays in fp16's normal range, and the epilogue multiplies the accumulators by 1 / wscale (exact).
    bool f16 = false;
    double wscale = 1.0;
    // int8 digit planes (ISB_PREC_I8X*): W_offdiag = q0 * sum_t 256^(P-1-t) digit_t, q0 a power of two; the diagonal of
    // a square model is kept apart (diag_d / diag_f, multiples of q0) and added by the epilogue
    bool i8 = false;
    double q0 = 1.0;
    bool i8_wide = false;    // every row's L1 norm (both orientations) < 2^31 quanta: the fast path recombines all planes in int32
    double *diag_d = nullptr;
    float *diag_f = nullptr;
    int ldkv = 0, ldkh = 0;            // K pitch (elements) of the two operand orientations
    __nv_bfloat16 *Wt[TC_PMAX] = {};   // hidden update operand: [nh][ldkv]  (K = visible units); int8 planes when i8
    __nv_bfloat16 *Wn[TC_PMAX] = {};   // visible update operand: [nv][ldkh] (K = hidden units)
    CUtensorMap mapWt[TC_PMAX], mapWn[TC_PMAX];
    int bn_h = 0, bn_v = 0;            // default tile widths for the hidden / visible update (least padding)
    int rows_t = 0, cols_t = 0, rows_n = 0, cols_n = 0;  // shapes of the two operand orientations
    struct BnMaps {
        int orient, bn;
        CUtensorMap m[TC_PMAX];
    };
    std::vector<BnMaps> bn_cache;      // tensor maps for other tile widths (the box height is part of the map)
    float *bias_hf = nullptr, *bias_vf = nullptr;  // hidden / visible biases in float, zero padded to 16
};
struct TcEns {
    // [R][ldkv], [R][ldkh] +-1 in the operand format; int8 mode: aliases of the ensemble's canonical int8 arrays
    __nv_bfloat16 *Sv = nullptr, *Sh = nullptr;
    bool alias = false;
    CUtensorMap mapSv, mapSh;
};

// One layer update (= one GEMM shape): which units are sampled, from which input layer
struct TcLayer {
    int nout, kin, bn, n_tiles, num_kb;
    int bn_mma;       // N of the MMA = rows of the coupling tile: bn, or P * bn for stacked int8 digit planes
    int u_off;        // global index of output unit 0 (row-sharded models: this rank's block offset), else 0
    int kb_per_blk;   // K blocks per slab of the A operand (block-major [G][R][nb] spin matrices), else num_kb
    void *out_bf;            // [R][ldo] the sampled layer in the operand format (bf16 / fp16 / int8 +-1; on entry: its
                             // previous values, read by MomentumAnnealing)
    int64_t ldo;
    // int8 mode, square models: diagonal couplings of this layer's units (NULL: none) and where unit u's own INPUT
    // spin of replica r lives: in_diag[r * ld_in + u] (int8)
    const float *diag_f;
    const double *diag_d;
    const int8_t *in_diag;
    int64_t ld_in;
    const double *bias;      // [nout]
    const float *bias_f;     // [nout rounded up to 16] the same in float (Philox mode)
    const double *F;         // external fluctuations (f64) or NULL
    uint32_t domain;         // Philox stream of this layer
    // fused all-gather (row-sharded SCA): the sampled block is also stored straight into every peer GPU's
    // gathered matrix through NVLink-mapped pointers (same [R][ldo] addressing as out_bf), tile by tile
    int npeer;
    void *peer[7];
};
struct TcParams {
    TcLayer L[2];     // [1] = hidden from visible, [0] = visible from hidden (persistent mode uses both)
    int R, P, rule, fluct_mode;
    // work decomposition.  persist == 0: one half-step (layer `layer`), tiles (m_blk, n_blk) strided over the grid.
    // persist == 1: chain-resident: CTA c owns the replicas [c*rows_per_cta, (c+1)*rows_per_cta) and runs
    // `nsteps_seg` full steps (hidden then visible) on them without leaving the SM — chains are independent, so
    // no grid-wide synchronisation exists; only the CTA's own producer waits for its own epilogue.
    int persist, layer, m_tiles, rows_per_cta, nsteps_seg;
    // cg = 2 always: the CTAs run in pairs (cta_group::2).  The two CTAs of a cluster run one M = 256 MMA together: CTA
    // `rank` owns the replicas [m0 + 128 rank, + 128) of the pair's tile and loads the rows [rank bn/2, + bn/2) of the
    // coupling tile, so every SM ingests half of W per tile.  m_tiles counts tiles of 128 cg replicas.
    int cg;
    // chain-resident mode: the epilogue publishes its progress through the layer it is writing (one mbarrier per
    // tile and per round of TC_GW columns, sig_gpt[layer] rounds per tile), and the producer of the next half-step
    // waits K block by K block instead of for the whole layer.  The last `sig_fine` tiles of a half-step (always 1)
    // publish after every round (one proxy fence each), the earlier tiles once at their end.
    // cg and sig_fine are parameters rather than constants because folding either one into the kernel changes the
    // register allocation and schedule of the instantiations that were measured.
    int sig_gpt[2], sig_fine;
    int r_off;               // global replica index of row 0 (a run may hold a slice of the replicas): Philox only
    uint32_t fmt;            // operand format: 0 bf16 terms, 1 fp16 terms, 2 int8 digit planes (selects the instantiation)
    float acc_scale;         // accumulator -> field: 1 / (power-of-two pre-scale of the fp16 couplings), 1 for bf16
    int i8_comb;             // int8 fast path: how the plane sums recombine (i8_field16): 0 per plane, 1 exact pairs, 2 all in int32
    float i8_sf[TC_PMAX];    // int8: weight of plane t, q0 * 256^(P-1-t) (powers of two), as float and as double
    double i8_sd[TC_PMAX];
    int64_t nsteps, k0;      // steps of the whole run (fluctuation array pitch), first step of this launch
    const double *Tsched;
    const double *tscale;    // per-replica temperature factors [R] or NULL
    int64_t steps_per_T;
    double T_direct;         // temperature when Tsched is NULL
    uint64_t seed, step_abs0;  // Philox step of k0
    PhiloxKeys keys;           // the ten round keys of `seed`, filled by the host: constant-bank operands of the Philox
                               // rounds instead of twenty registers of every sampling thread
};

// The tile jobs of a CTA, enumerated identically by the producer, the MMA issuer and the epilogue warps.
struct TcJob {
    int layer, m0, n_blk, hs;   // hs = half-step index within the launch (0 when !persist)
    int64_t k;                  // step index within the run
    bool hs_first, hs_last;
};
struct TcJobIter {
    int tile, layer, n_blk, step, crank;
    __device__ __forceinline__ void init(const TcParams &p, int cta_rank_in_pair) {
        tile = blockIdx.x / p.cg;
        crank = cta_rank_in_pair;
        layer = 1;
        n_blk = 0;
        step = 0;
    }
    __device__ __forceinline__ bool next(const TcParams &p, TcJob &j) {
        if (!p.persist) {
            const int nt = p.L[p.layer].n_tiles;
            if (tile >= p.m_tiles * nt) return false;
            j.layer = p.layer;
            j.m0 = (tile / nt) * (TC_BM * p.cg) + crank * TC_BM;
            j.n_blk = tile % nt;
            j.hs = 0;
            j.k = p.k0;
            j.hs_first = j.hs_last = false;
            tile += gridDim.x / p.cg;
            return true;
        }
        if (step >= p.nsteps_seg) return false;
        j.layer = layer;
        j.m0 = blockIdx.x * p.rows_per_cta;
        j.n_blk = n_blk;
        j.hs = 2 * step + (layer == 1 ? 0 : 1);
        j.k = p.k0 + step;
        j.hs_first = n_blk == 0;
        j.hs_last = n_blk == p.L[layer].n_tiles - 1;
        if (++n_blk == p.L[layer].n_tiles) {
            n_blk = 0;
            if (layer == 1) {
                layer = 0;
            } else {
                layer = 1;
                ++step;
            }
        }
        return true;
    }
};

// ------------------------------------------------------------------ PTX wrappers (tcgen05 / TMA)
// All of them act for a CTA pair (the two CTAs of a cluster on one TPC): each CTA loads its own A rows and HALF of
// the B tile; the bytes of both CTAs complete on the leader's (cluster rank 0) full barrier, whose address
// `leader_bar` is a shared::cluster address obtained with mapa.
__device__ __forceinline__ uint32_t mapa_rank0(const void *smem_ptr) {
    uint32_t ra;
    asm volatile("mapa.shared::cluster.u32 %0, %1, 0;" : "=r"(ra) : "r"(smem_u32(smem_ptr)));
    return ra;
}
// Arrive on the leader's barrier (a shared::cluster address from mapa_rank0).  No .release.cluster here: the arrivals
// this kernel sends to the peer order nothing the generic proxy wrote (TMA bytes are tracked by complete_tx, TMEM reads
// are fenced by tcgen05.fence), and a cluster-scope release per ring slot throttled the producer loop.
__device__ __forceinline__ void mbar_arrive_cluster_addr(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void *smem_dst, const CUtensorMap *map, int c0, int c1, uint32_t leader_bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
            smem_u32(smem_dst)),
        "l"(map), "r"(leader_bar), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_3d(void *smem_dst, const CUtensorMap *map, int c0, int c1, int c2, uint32_t leader_bar) {
    asm volatile(
        "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
            smem_u32(smem_dst)),
        "l"(map), "r"(leader_bar), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t *smem_slot, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_slot)), "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// true in exactly one (converged) lane of the warp
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// issued by the leader CTA only: M = 256 (128 rows of A per CTA), each CTA holds half of B's rows
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
        : "memory");
}
// kind::i8: A, B signed 8-bit, D = int32 accumulators, K = 32 per instruction (the same 32 operand bytes per row)
__device__ __forceinline__ void umma_i8(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
        : "memory");
}
// the arrive is multicast to the barrier at the same offset in both CTAs of the pair
__device__ __forceinline__ void umma_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                     smem_u32(bar)),
                 "h"((uint16_t)3)
                 : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
// the same load without the wait: several loads in flight, one tmem_ld_wait() before the first use
__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// K-major, 128B-swizzled operand tile (rows x 64 bf16): SBO = 1024 B (8 rows), LBO = 1 (unused), version 1.
__device__ __forceinline__ uint64_t umma_desc_sw128(const void *smem_tile) {
    const uint32_t lo = ((smem_u32(smem_tile) >> 4) & 0x3FFFu) | (1u << 16);
    const uint32_t hi = (1024u >> 4) | (1u << 14) | (2u << 29);
    return ((uint64_t)hi << 32) | lo;
}
// kind::f16 instruction descriptor: D = f32 (bit 4), A / B format at bits 7 / 10 (0 = fp16, 1 = bf16), both K-major,
// M = m (128, or 256 for a CTA pair), N = bn
__device__ __forceinline__ uint32_t umma_idesc_bf16(int m, int bn, uint32_t f16) {
    const uint32_t fmt = f16 ? 0u : 1u;
    return (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(bn >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
// kind::i8 instruction descriptor: D = s32 (c_format 2 at bit 4), A / B = signed 8-bit (1 at bits 7 / 10), K-major
__device__ __forceinline__ uint32_t umma_idesc_i8(int m, int bn) {
    return (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(bn >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// int8 digit planes, fast sampling path: the fields of 16 units from their P exact int32 plane sums.  On entry xf holds the
// biases.  COMB = 2 (P = 3): the planes recombine EXACTLY in int32, (v0 2^8 + v1) 2^8 + v2 — the model builder checked that
// every row's L1 norm stays below 2^31 quanta — one conversion and one FFMA per unit; COMB = 1: exact pairs 2^8 v_2i + v_2i+1
// (|.| <= 32896 K < 2^31 for the K <= 65000 the host admits); COMB = 0: one conversion and one FFMA per plane.  The unsigned
// shifts wrap modulo 2^32, which is the exact two's-complement result whenever the true value fits.
template <int P, int COMB>
__device__ __forceinline__ void i8_field16(uint32_t tq, uint32_t pstride, const float *sf, float (&xf)[16]) {
    if constexpr (COMB == 0) {
#pragma unroll
        for (int t = 0; t < P; ++t) {
            uint32_t v[16];
            tmem_ld16(tq + (uint32_t)t * pstride, v);
#pragma unroll
            for (int j = 0; j < 16; ++j) xf[j] = fmaf((float)(int)v[j], sf[t], xf[j]);
        }
    } else {
        uint32_t hi[16], v1[16];
        tmem_ld16_nowait(tq, hi);
        tmem_ld16_nowait(tq + pstride, v1);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 16; ++j) hi[j] = (hi[j] << 8) + v1[j];
        if constexpr (P == 2) {
#pragma unroll
            for (int j = 0; j < 16; ++j) xf[j] = fmaf((float)(int)hi[j], sf[1], xf[j]);
        } else if constexpr (P == 3) {
            tmem_ld16(tq + 2u * pstride, v1);
            if constexpr (COMB == 2) {
#pragma unroll
                for (int j = 0; j < 16; ++j) xf[j] = fmaf((float)(int)((hi[j] << 8) + v1[j]), sf[2], xf[j]);
            } else {
#pragma unroll
                for (int j = 0; j < 16; ++j) xf[j] = fmaf((float)(int)hi[j], sf[1], fmaf((float)(int)v1[j], sf[2], xf[j]));
            }
        } else {
            uint32_t lo[16];
            tmem_ld16_nowait(tq + 2u * pstride, lo);
            tmem_ld16_nowait(tq + 3u * pstride, v1);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 16; ++j)
                xf[j] = fmaf((float)(int)hi[j], sf[1], fmaf((float)(int)((lo[j] << 8) + v1[j]), sf[3], xf[j]));
        }
    }
}

#ifdef ISB_TC_TIMING   // measurement build only (scripts/tc_timing.py): where the sampling warps' cycles go
__device__ long long g_tc_timing[296 * 16 * 4];
#define TC_TIME(var) const long long var = clock64()
#else
#define TC_TIME(var)
#endif
// ------------------------------------------------------------------ the kernel
__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ void fence_proxy_async_global() { asm volatile("fence.proxy.async.global;" ::: "memory"); }

// Every wait of the kernel polls (mbar_wait).  The barriers complete through the peer CTA (remote arrives, multicast
// commits, the peer's TMA bytes), and suspended waits (a try_wait time hint) gained nothing there (DESIGN §3).  The
// producer and the MMA issuer are one thread each: polling costs two threads' issue slots, and the dependency chain
// epilogue -> producer -> TMA -> MMA of a half-step boundary carries no wake-up latency.

struct TcMaps {
    CUtensorMap A[2];     // input spin matrix of layer update [1] (visible layer) and [0] (hidden layer)
    CUtensorMap B[2][TC_PMAX];  // coupling terms / digit planes of the two orientations
};

// FMT: operand format (0 bf16 terms, 1 fp16 terms of the pre-scaled couplings, 2 int8 digit planes); a template
// parameter, so that the bf16 instantiations keep their code (and registers) exactly.
template <bool EXTF, int FMT>
__global__ void __launch_bounds__(TC_THREADS, 1) bip_tc_kernel(const __grid_constant__ TcMaps maps, const TcParams p) {
    constexpr bool F16 = FMT == 1;
    constexpr bool I8 = FMT == 2;
    constexpr int BK = I8 ? TC_BK8 : TC_BK;                   // K elements per ring slot (128 bytes either way)
    constexpr uint32_t ONE2 = F16 ? 0x3C003C00u : 0x3F803F80u;  // two packed +1 of the operand format
    constexpr int NST = TC_STAGES;                            // ring slots
    constexpr int STB = TC_STAGE_BYTES;                       // bytes per slot
    extern __shared__ unsigned char smem_dyn[];
    unsigned char *smem = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~(uintptr_t)1023);
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + (size_t)TC_STAGES * TC_STAGE_BYTES);
    uint64_t *full_bar = bars;                     // [NST]
    uint64_t *empty_bar = bars + NST;        // [NST]
    uint64_t *tfull_bar = bars + 2 * NST;    // [2]
    uint64_t *tempty_bar = bars + 2 * NST + 2;  // [2] (two accumulator stages)
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2 * NST + 7);
    uint64_t *sig_bar = bars + 2 * NST + 8;  // [2][TC_SIG_MAX] chain-resident mode: epilogue -> producer progress

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int crank = (int)cluster_ctarank();  // rank in the CTA pair; 0 = leader (issues the MMAs)
    const bool leader = crank == 0;

    if (threadIdx.x == 0) {
        for (int s = 0; s < NST; ++s) {
            mbar_init(&full_bar[s], 2);   // the leader's barrier takes one arrive per CTA and both CTAs' bytes
            mbar_init(&empty_bar[s], 1);
        }
        for (int a = 0; a < 2; ++a) mbar_init(&tfull_bar[a], 1);
        for (int a = 0; a < 2; ++a)
            mbar_init(&tempty_bar[a], 2 * TC_EPI_WARPS);  // the epilogue warps of both CTAs release the leader's
        if (p.persist)
            for (int i = 0; i < 2 * TC_SIG_MAX; ++i) mbar_init(&sig_bar[i], TC_EPI_WARPS);
        mbar_fence_init();
    }
    if (warp == 2) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    // no remote arrive, multicast commit or 2-CTA MMA may touch the peer before its barriers / TMEM exist
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    TcJobIter jobs;
    jobs.init(p, crank);
    TcJob job;

    if (warp < 4) {
    if (warp == 0) {
        // ================================================================ TMA producer
        // (the whole warp walks the loop, one elected lane issues: see the MMA issuer below)
        {
            int s = 0;            // ring slot and its phase, kept incrementally
            uint32_t ph = 0;
            while (jobs.next(p, job)) {
                const TcLayer &L = p.L[job.layer];
                // chain-resident mode: this half-step's A operand is what the CTA's own epilogue wrote during the
                // previous half-step (generic-proxy stores, fenced to the async proxy before the arrive).  Only the
                // first tile of a half-step can run into it; K block kb needs the input units [64 kb, 64 kb + 64).
                const bool dep = p.persist && job.hs_first && job.hs > 0;
                const int pl = 1 - job.layer;   // the layer sampled by the previous half-step = this one's input
                const uint32_t dep_par = (uint32_t)((job.hs >> 1) - (job.layer == 1 ? 1 : 0)) & 1u;
                int waited = -1;
                const int bnc = L.bn_mma / 2;  // rows of the coupling tile this CTA loads
                const uint32_t tx = (uint32_t)(TC_A_BYTES + bnc * 128);
                const int num_kb = L.num_kb;
                // 16-bit terms: K block outer, term inner (all terms accumulate into one accumulator).  int8 digit
                // planes: one stacked coupling tile per K block (all planes in one MMA).
                const int n_inner = I8 ? 1 : p.P;
                {
                int kq = 0, kr = 0;             // kb = kq * kb_per_blk + kr (slab of the A operand, block within it)
                for (int kb = 0; kb < num_kb; ++kb) {
                    if (dep) {
                        const int ul = min(kb * BK + BK - 1, p.L[pl].nout - 1);
                        const int idx = (ul / p.L[pl].bn) * p.sig_gpt[pl] + (ul % p.L[pl].bn) / TC_GW;
                        if (idx > waited) {
                            mbar_wait(&sig_bar[pl * TC_SIG_MAX + idx], dep_par);
                            waited = idx;
                        }
                    }
                    for (int ti = 0; ti < n_inner; ++ti) {
                        const int t = ti;
                        mbar_wait(&empty_bar[s], ph ^ 1u);
                        unsigned char *sa = smem + (size_t)s * STB;
                        if (elect_one()) {
                            const uint32_t lbar = mapa_rank0(&full_bar[s]);
                            if (leader)
                                mbar_arrive_expect_tx(&full_bar[s], 2u * tx);
                            else
                                mbar_arrive_cluster_addr(lbar);
                            tma_load_3d(sa, &maps.A[job.layer], kr * BK, job.m0, kq, lbar);
                            tma_load_2d(sa + TC_A_BYTES, &maps.B[job.layer][t], kb * BK, job.n_blk * L.bn_mma + crank * bnc, lbar);
                        }
                        __syncwarp();
                        if (++s == NST) {
                            s = 0;
                            ph ^= 1u;
                        }
                    }
                    if (++kr == L.kb_per_blk) {
                        kr = 0;
                        ++kq;
                    }
                }
                }
            }
            // the leader's commits also arrive on this CTA's empty barriers: do not retire (or let the peer retire)
            // before the last of them has landed
            for (int i = 0; i < NST; ++i) {
                mbar_wait(&empty_bar[s], ph ^ 1u);
                if (++s == NST) {
                    s = 0;
                    ph ^= 1u;
                }
            }
        }
    } else if (warp == 1) {
        // ================================================================ MMA issuer (the leader CTA's only)
        // The WHOLE warp walks this loop and one elected lane issues: with warp-uniform control flow the smem
        // descriptors, TMEM and barrier addresses stay in uniform registers.  (Under `if (lane == 0)` ptxas wrapped every
        // tcgen05 instruction in an ELECT / R2UR.BROADCAST / BRA.U.ANY loop: 112 instructions per K block, 890 cycles for
        // 512 cycles of MMA — the issuing thread, not the operand feed, bounded the contraction.)
        if (leader) {
            uint32_t tl = 0;
            int s = 0;            // ring slot and its phase, kept incrementally
            uint32_t ph = 0;
            const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
            while (jobs.next(p, job)) {
                const TcLayer &L = p.L[job.layer];
                const uint32_t idesc = I8 ? umma_idesc_i8(2 * TC_BM, L.bn_mma) : umma_idesc_bf16(2 * TC_BM, L.bn_mma, F16 ? 1u : 0u);
                const int num_kb = L.num_kb;
                const int a = tl & 1;
                // one accumulator stage per tile: all K blocks x terms (16-bit), or the stacked planes (int8), into it
                const int iters = I8 ? num_kb : num_kb * p.P;
                // the last K block of a layer may hold fewer than 4 x 32 bytes of real input units (K = 784: 16 of 128): the
                // rest of the slot is zero fill, its MMAs are skipped.  (No division in the issue loop: it is the kernel's
                // critical thread, see above.)
                const int i_tail = L.kb_per_blk == L.num_kb ? iters - (I8 ? 1 : p.P) : iters;   // first iteration of the last K block
                const int nk_tail = min(4, (L.kin - (num_kb - 1) * BK + BK / 4 - 1) / (BK / 4));
                {
                    mbar_wait(&tempty_bar[a], ((tl >> 1) & 1) ^ 1);  // epilogue has drained this accumulator
                    const uint32_t d_tmem = tmem_u + (uint32_t)(a * TC_BN_MAX);
                    tc_fence_after();
                    for (int i = 0; i < iters; ++i) {
                        mbar_wait(&full_bar[s], ph);
                        tc_fence_after();
                        const unsigned char *sa = smem + (size_t)s * STB;
                        const uint64_t adesc = umma_desc_sw128(sa);
                        const uint64_t bdesc = umma_desc_sw128(sa + TC_A_BYTES);
                        const int nk = i >= i_tail ? nk_tail : 4;
                        if (elect_one()) {
                            if (nk == 4) {   // (the common block, kept as four back-to-back issues)
#pragma unroll
                                for (int k = 0; k < 4; ++k) {  // 4 x 32 operand bytes per slot row: advance 2 descriptor units along K
                                    if constexpr (I8)
                                        umma_i8(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (i | k) ? 1u : 0u);
                                    else
                                        umma_bf16(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (i | k) ? 1u : 0u);
                                }
                            } else {
                                for (int k = 0; k < nk; ++k) {
                                    if constexpr (I8)
                                        umma_i8(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (i | k) ? 1u : 0u);
                                    else
                                        umma_bf16(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (i | k) ? 1u : 0u);
                                }
                            }
                            umma_commit(&empty_bar[s]);  // slot free (in both CTAs) when these MMAs have read it
                        }
                        __syncwarp();
                        if (++s == NST) {
                            s = 0;
                            ph ^= 1u;
                        }
                    }
                }
                if (elect_one()) umma_commit(&tfull_bar[a]);  // accumulator complete (each CTA: its 128 replicas x bn units)
                __syncwarp();
                ++tl;
            }
        }
    }
    } else {
        // ================================================================ epilogue (sampling rule)
        const int ew = warp - 4;
        const int quad = warp & 3;          // TMEM lane quadrant this warp may read: lanes 32*(warpid % 4) ..
        const int half = ew >> 2;           // the warps of a quadrant interleave the 16-column chunks
        const PhiloxKeys &keys = p.keys;
        uint32_t tl = 0;
        int rot = 0;                        // tl % TC_HALVES, kept incrementally
#ifdef ISB_TC_TIMING
        long long tm_wait = 0, tm_chunk = 0, tm_post = 0;
        const long long tm_start = clock64();
#endif
        // Temperature-derived constants of this thread's replica.  In chain-resident mode they change once per step (the
        // replica of a thread is fixed), so the schedule load (an L2 round trip), the 64-bit division and the float
        // reciprocal run once per half-step instead of once per tile: with K <= 784 a tile is only 64-80 units wide, and
        // this per-tile prologue was 40 % of the sampling warps' instructions (ncu, profiles/r2o_c4_i8x3_ncu_summary.txt).
        double Td = 0.0;
        float Tf = 0.f, cS = 0.f, cE = 0.f;
        bool fast_hs = false;
        // One tile of layer LY.  The layer index is a compile-time constant (two copies of the tile code): every field of
        // p.L[LY] is then a direct constant-bank operand instead of an indexed LDC with its scoreboard wait — the per-tile
        // prologue of the 64-80 unit tiles of config 4 was a fifth of the sampling warps' time (ncu source page).
        auto epi_tile = [&](auto lyc) {
            constexpr int LY = decltype(lyc)::value;
            const TcLayer &L = p.L[LY];
            const uint64_t step_abs = p.step_abs0 + (uint64_t)(job.k - p.k0);
            constexpr int CW = TC_CW;
            const int nchunks = L.bn / CW;
            const int a = tl & 1;
            // the warps of a quadrant take the chunks of a round in an order that rotates from tile to tile: when a
            // tile's last round has fewer chunks than warps, a different warp goes ahead to the next tile each time
            const int hrot = half + rot >= TC_HALVES ? half + rot - TC_HALVES : half + rot;
            const int lrow = quad * 32 + lane;
            const int r = job.m0 + lrow;
            const bool row_ok = r < p.R && (!p.persist || lrow < p.rows_per_cta);
            if (!p.persist || job.hs_first) {
                // temperature of this thread's replica (per-replica factors make it a per-row quantity); fetched BEFORE
                // the wait for the accumulator, so that the schedule load overlaps the MMAs
                Td = p.Tsched ? __ldg(&p.Tsched[job.k / p.steps_per_T]) : p.T_direct;
                if (p.tscale && row_ok) Td = __dmul_rn(Td, __ldg(&p.tscale[r]));
                Tf = (float)Td;
                cS = 0.5f * Tf * 0.69314718055994531f;  // (T/2) ln 2
                cE = Tf > 0.f ? -2.0f * 1.4426950408889634f / Tf : 0.f;  // e^{-2x/T} = 2^{cE x}
                // Fast path for the common case (SCA, in-kernel noise, every replica of the warp at T > 0, no peer copies,
                // a chunk of CW real units): a branch-free body with everything tile-invariant hoisted.  The rule is
                // evaluated with three fma-pipe operations per unit:
                //   u (1 + e^{-2x/T}) > 1,  u = (w + 1/2) 2^-32    <=>    (float)w (1 + 2^{cE x}) > 2^32
                // (x = acc + bias: FADD; cE x: FMUL; the left side: one FFMA; the compare and the sign packing run on the
                // ALU pipe, the conversion and the exponential on the XU).
                fast_hs = !EXTF && p.rule == ISB_BIP_SCA && L.npeer == 0 && !__any_sync(0xFFFFFFFFu, !(Tf > 0.f));
            }
            TC_TIME(tw0);
            mbar_wait(&tfull_bar[a], (tl >> 1) & 1);
            tc_fence_after();
            TC_TIME(tw1);
            const int gpt = p.sig_gpt[LY];
            const bool fine = p.persist && job.n_blk >= L.n_tiles - p.sig_fine;
            uint64_t *sig = sig_bar + LY * TC_SIG_MAX + job.n_blk * gpt;
            const bool fastp = fast_hs;
            const int tile_u0 = job.n_blk * L.bn;
            const int nfull = fastp ? min(L.bn, L.nout - tile_u0) / CW : 0;   // chunks the fast path takes
            const float *bias_t = L.bias_f + tile_u0;
            const uint32_t taddr_t = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(a * TC_BN_MAX);
            const uint32_t pc2 = (uint32_t)(r + p.r_off), pc3 = (L.domain << 28) | (uint32_t)((L.u_off + tile_u0) >> 2);
            if constexpr (I8) {
              // ---- int8 digit planes: P exact int32 accumulators per unit, recombined here
              const int rr = row_ok ? r : job.m0;   // rows without a replica read / compute on a valid row, store nothing
              int8_t *out8 = reinterpret_cast<int8_t *>(L.out_bf) + (int64_t)rr * L.ldo + tile_u0;
              const int8_t *in8 = L.in_diag ? L.in_diag + (int64_t)rr * L.ld_in + tile_u0 : nullptr;
              const uint32_t tq = taddr_t;          // plane t of the tile: columns [t * bn, (t + 1) * bn) of stage a
              const uint32_t pstride = (uint32_t)L.bn;
              for (int g = 0; g * TC_HALVES < nchunks; ++g) {
                const int c = g * TC_HALVES + hrot;
                if (c < nfull) {
                  // fast path (SCA, in-kernel noise, T > 0, 16 real units): field in float — every plane sum is an exact
                  // integer and every plane weight a power of two (i8_field16: the planes are recombined in int32 where that is exact)
                  float xf[16];
#pragma unroll
                  for (int q = 0; q < 4; ++q) {
                      const float4 b4 = __ldg(reinterpret_cast<const float4 *>(bias_t + c * 16) + q);
                      xf[4 * q] = b4.x; xf[4 * q + 1] = b4.y; xf[4 * q + 2] = b4.z; xf[4 * q + 3] = b4.w;
                  }
                  {
                      const uint32_t tc0 = tq + (uint32_t)(c * 16);
                      const int form = p.i8_comb * 8 + p.P;   // warp-uniform (kernel parameters); a chain of uniform
                      if (form == 2 * 8 + 3)                   // branches, the common forms first (a jump table costs an
                          i8_field16<3, 2>(tc0, pstride, p.i8_sf, xf);   // indirect branch per chunk)
                      else if (form == 1 * 8 + 3)
                          i8_field16<3, 1>(tc0, pstride, p.i8_sf, xf);
                      else if (form == 1 * 8 + 2)
                          i8_field16<2, 1>(tc0, pstride, p.i8_sf, xf);
                      else if (form == 1 * 8 + 4)
                          i8_field16<4, 1>(tc0, pstride, p.i8_sf, xf);
                      else if (form == 0 * 8 + 2)
                          i8_field16<2, 0>(tc0, pstride, p.i8_sf, xf);
                      else if (form == 0 * 8 + 3)
                          i8_field16<3, 0>(tc0, pstride, p.i8_sf, xf);
                      else
                          i8_field16<4, 0>(tc0, pstride, p.i8_sf, xf);
                  }
                  if (in8) {  // the unit's own coupling (square models): diag * own input spin
                      const uint4 sv = __ldcg(reinterpret_cast<const uint4 *>(in8 + c * 16));
                      const uint32_t sw[4] = {sv.x, sv.y, sv.z, sv.w};
#pragma unroll
                      for (int q = 0; q < 4; ++q) {
                          const float4 d4 = __ldg(reinterpret_cast<const float4 *>(L.diag_f + tile_u0 + c * 16) + q);
                          const float dd[4] = {d4.x, d4.y, d4.z, d4.w};
#pragma unroll
                          for (int e = 0; e < 4; ++e)
                              xf[4 * q + e] += ((sw[q] >> (8 * e + 7)) & 1u) ? -dd[e] : dd[e];
                      }
                  }
                  Philox4 blk[4];
#pragma unroll
                  for (int q = 0; q < 4; ++q)
                      blk[q] = philox4x32_10k((uint32_t)step_abs, (uint32_t)(step_abs >> 32), pc2, pc3 + (uint32_t)(c * 4 + q), keys);
                  uint32_t wb[4] = {0x01010101u, 0x01010101u, 0x01010101u, 0x01010101u};
#pragma unroll
                  for (int j = 0; j < 16; ++j) {
                      const float wf = (float)philox_pick(blk[j >> 2], (uint32_t)(j & 3));
                      if (fmaf(wf, ex2_approx(cE * xf[j]), wf) > 4294967296.0f) wb[j >> 2] |= 0xFEu << (8 * (j & 3));
                  }
                  if (row_ok) *reinterpret_cast<uint4 *>(out8 + c * 16) = make_uint4(wb[0], wb[1], wb[2], wb[3]);
                } else if (c < nchunks && tile_u0 + c * 16 < L.nout) do {   // (chunks of padding units: nothing to do)
                  // general path: the field in double, EXACT (every term is a multiple of the quantum q0)
                  double xd[16];
#pragma unroll
                  for (int j = 0; j < 16; ++j) xd[j] = 0.0;
                  for (int t = 0; t < p.P; ++t) {
                      uint32_t v[16];
                      tmem_ld16(tq + (uint32_t)t * pstride + (uint32_t)(c * 16), v);
                      const double sd = p.i8_sd[t];
#pragma unroll
                      for (int j = 0; j < 16; ++j) xd[j] = fma((double)(int)v[j], sd, xd[j]);
                  }
                  const int u0 = tile_u0 + c * 16;
                  if (!row_ok || u0 >= L.nout) break;
                  int8_t *ob = out8 + c * 16;
                  const bool full = u0 + 16 <= L.nout;
                  uint32_t wb[4] = {0x01010101u, 0x01010101u, 0x01010101u, 0x01010101u};
#pragma unroll
                  for (int j = 0; j < 16; ++j) {
                      const int u = u0 + j;
                      if (u >= L.nout) continue;
                      if (in8) xd[j] += (__ldcg(in8 + c * 16 + j) < 0) ? -L.diag_d[u] : L.diag_d[u];
                      const bool old_neg = p.rule == ISB_BIP_MA && ob[j] < 0;  // MomentumAnnealing: own previous value
                      bool neg;
                      if (EXTF) {
                          const double f = p.fluct_mode == ISB_FLUCT_SHARED ? L.F[job.k * L.nout + u]
                                                                             : L.F[((int64_t)r * p.nsteps + job.k) * L.nout + u];
                          double ft = __dmul_rn(f, Td);
                          if (p.rule == ISB_BIP_MA && old_neg) ft = -ft;
                          neg = __dsub_rn(__dmul_rn(2.0, __dadd_rn(xd[j], L.bias[u])), ft) < 0.0;
                      } else {
                          const Philox4 b4 = philox4x32_10k((uint32_t)step_abs, (uint32_t)(step_abs >> 32), (uint32_t)(r + p.r_off),
                                                            (L.domain << 28) | (uint32_t)((L.u_off + u) >> 2), keys);
                          const uint32_t w = philox_pick(b4, (uint32_t)((L.u_off + u) & 3));
                          const float x = (float)xd[j] + L.bias_f[u];
                          const float uu = fmaf((float)w, 2.3283064365386963e-10f, 1.1641532182693481e-10f);  // (w+1/2) 2^-32
                          float tt;
                          if (Tf == 0.f) {
                              tt = x + 0.0f;
                          } else if (p.rule == ISB_BIP_SCA) {
                              tt = 1.0f - fmaf(uu, ex2_approx(cE * x), uu);
                          } else {
                              const float l = cS * __log2f(uu);
                              tt = x + (old_neg ? -l : l);
                          }
                          neg = (__float_as_uint(tt) & 0x80000000u) != 0u;
                      }
                      if (neg) wb[j >> 2] |= 0xFEu << (8 * (j & 3));
                  }
                  if (full) {
                      *reinterpret_cast<uint4 *>(ob) = make_uint4(wb[0], wb[1], wb[2], wb[3]);
                      for (int pq = 0; pq < L.npeer; ++pq)  // peer stores over NVLink overlap the next tile's MMAs
                          *reinterpret_cast<uint4 *>(reinterpret_cast<int8_t *>(L.peer[pq]) + (int64_t)r * L.ldo + u0) =
                              make_uint4(wb[0], wb[1], wb[2], wb[3]);
                  } else {
                      for (int j = 0; j < 16 && u0 + j < L.nout; ++j) ob[j] = (int8_t)((wb[j >> 2] >> (8 * (j & 3))) & 0xFFu);
                  }
                } while (0);
                if (fine) {
                  fence_proxy_async_global();
                  __syncwarp();
                  if (lane == 0) mbar_arrive(&sig[g]);
                }
              }
            } else {
            __nv_bfloat16 *out_t = reinterpret_cast<__nv_bfloat16 *>(L.out_bf) + (int64_t)(row_ok ? r : job.m0) * L.ldo + tile_u0;
            for (int g = 0; g * TC_HALVES < nchunks; ++g) {
              const int c = g * TC_HALVES + hrot;
              if (c < nfull) {
                uint32_t v[16];
                tmem_ld16(taddr_t + (uint32_t)(c * 16), v);
                float bf[16];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const float4 b4 = __ldg(reinterpret_cast<const float4 *>(bias_t + c * 16) + q);
                    bf[4 * q] = b4.x; bf[4 * q + 1] = b4.y; bf[4 * q + 2] = b4.z; bf[4 * q + 3] = b4.w;
                }
                Philox4 blk[4];
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    blk[q] = philox4x32_10k((uint32_t)step_abs, (uint32_t)(step_abs >> 32), pc2, pc3 + (uint32_t)(c * 4 + q), keys);
                uint32_t wb[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) wb[j] = ONE2;
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const float wf = (float)philox_pick(blk[j >> 2], (uint32_t)(j & 3));
                    const float x = F16 ? fmaf(__uint_as_float(v[j]), p.acc_scale, bf[j]) : __uint_as_float(v[j]) + bf[j];
                    if (fmaf(wf, ex2_approx(cE * x), wf) > 4294967296.0f) wb[j >> 1] |= 0x8000u << (16 * (j & 1));
                }
                if (row_ok) {
                    uint4 *o = reinterpret_cast<uint4 *>(out_t + c * 16);
                    o[0] = make_uint4(wb[0], wb[1], wb[2], wb[3]);
                    o[1] = make_uint4(wb[4], wb[5], wb[6], wb[7]);
                }
              } else if (c < nchunks) do {
                uint32_t v[CW];
                tmem_ld16(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(a * TC_BN_MAX + c * CW), v);
                const int u0 = job.n_blk * L.bn + c * CW;
                if (!row_ok || u0 >= L.nout) break;
                __nv_bfloat16 *ob = reinterpret_cast<__nv_bfloat16 *>(L.out_bf) + (int64_t)r * L.ldo + u0;
                const bool full = u0 + CW <= L.nout;
                // MomentumAnnealing multiplies the noise by the unit's own previous value: it is still in the
                // output matrix (bf16 +-1; pad columns read as 0 and are never stored)
                uint32_t oldw[CW / 2];
#pragma unroll
                for (int j = 0; j < CW / 2; ++j) oldw[j] = 0;
                if (p.rule == ISB_BIP_MA) {
#pragma unroll
                    for (int q = 0; q < CW / 8; ++q) {
                        const uint4 o = *reinterpret_cast<const uint4 *>(ob + 8 * q);
                        oldw[4 * q] = o.x; oldw[4 * q + 1] = o.y; oldw[4 * q + 2] = o.z; oldw[4 * q + 3] = o.w;
                    }
                }
                uint32_t wb[CW / 2];  // packed +-1 of the operand format = (0x3F80 | 0x3C00) | sign
#pragma unroll
                for (int j = 0; j < CW / 2; ++j) wb[j] = ONE2;
                if (EXTF) {
#pragma unroll
                    for (int j = 0; j < CW; ++j) {
                        const int u = u0 + j;
                        double x = 0.0;
                        if (u < L.nout) {
                            const double f = p.fluct_mode == ISB_FLUCT_SHARED ? L.F[job.k * L.nout + u]
                                                                               : L.F[((int64_t)r * p.nsteps + job.k) * L.nout + u];
                            double ft = __dmul_rn(f, Td);
                            if (p.rule == ISB_BIP_MA) ft = ((oldw[j >> 1] >> (16 * (j & 1) + 15)) & 1u) ? -ft : ft;
                            // (the accumulator times a power of two is exact)
                            const float accf = F16 ? __uint_as_float(v[j]) * p.acc_scale : __uint_as_float(v[j]);
                            x = __dsub_rn(__dmul_rn(2.0, __dadd_rn((double)accf, L.bias[u])), ft);
                        }
                        if (x < 0.0) wb[j >> 1] |= 0x8000u << (16 * (j & 1));
                    }
                } else {
                    float bf[CW];
                    if (full) {
#pragma unroll
                        for (int q = 0; q < CW / 4; ++q) {
                            const float4 b4 = __ldg(reinterpret_cast<const float4 *>(L.bias_f + u0) + q);
                            bf[4 * q] = b4.x; bf[4 * q + 1] = b4.y; bf[4 * q + 2] = b4.z; bf[4 * q + 3] = b4.w;
                        }
                    } else {
#pragma unroll
                        for (int j = 0; j < CW; ++j) bf[j] = u0 + j < L.nout ? __ldg(L.bias_f + u0 + j) : 0.f;
                    }
                    // the chunk's noise words first, in one branch-free block: the CW/4 Philox calls are independent
                    // dependency chains (IMAD.WIDE -> LOP3 -> IMAD.WIDE ...) that only overlap when they are adjacent
                    Philox4 blk[CW / 4];
#pragma unroll
                    for (int q = 0; q < CW / 4; ++q) {
                        // == philox_unit_block(seed, domain, r, step, unit >> 2) with the round keys hoisted
                        blk[q] = philox4x32_10k((uint32_t)step_abs, (uint32_t)(step_abs >> 32), (uint32_t)(r + p.r_off),
                                                (L.domain << 28) | (uint32_t)(((L.u_off + u0) >> 2) + q), keys);
                    }
#pragma unroll
                    for (int q = 0; q < CW / 4; ++q) {
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const int j = q * 4 + e;
                            const uint32_t w = philox_pick(blk[q], (uint32_t)e);
                            const float x = F16 ? fmaf(__uint_as_float(v[j]), p.acc_scale, bf[j]) : __uint_as_float(v[j]) + bf[j];
                            const float u = fmaf((float)w, 2.3283064365386963e-10f, 1.1641532182693481e-10f);  // (w+1/2) 2^-32
                            float t;
                            if (Tf == 0.f) {
                                t = x + 0.0f;  // no noise: sgn+(x); the addition turns a -0 accumulator into +0 (tie -> +1)
                            } else if (p.rule == ISB_BIP_SCA) {
                                // 2x - T ln(u/(1-u)) >= 0  <=>  u (1 + e^{-2x/T}) <= 1   (one MUFU.EX2)
                                t = 1.0f - fmaf(u, ex2_approx(cE * x), u);
                            } else {
                                // 2x - (-ln u) T s_old >= 0  <=>  x + (T/2) ln(u) s_old >= 0
                                const float l = cS * __log2f(u);
                                t = x + (((oldw[j >> 1] >> (16 * (j & 1) + 15)) & 1u) ? -l : l);
                            }
                            // sign bit of t (t is never NaN: u > 0, x finite; -0 cannot arise) -> sign bit of the bf16
                            wb[j >> 1] |= (j & 1) ? (__float_as_uint(t) & 0x80000000u) : ((__float_as_uint(t) & 0x80000000u) >> 16);
                        }
                    }
                }
                if (full) {
#pragma unroll
                    for (int q = 0; q < CW / 8; ++q)
                        *reinterpret_cast<uint4 *>(ob + 8 * q) = make_uint4(wb[4 * q], wb[4 * q + 1], wb[4 * q + 2], wb[4 * q + 3]);
                    for (int pq = 0; pq < L.npeer; ++pq) {  // peer stores over NVLink overlap the next tile's MMAs
                        __nv_bfloat16 *pb = reinterpret_cast<__nv_bfloat16 *>(L.peer[pq]) + (int64_t)r * L.ldo + u0;
#pragma unroll
                        for (int q = 0; q < CW / 8; ++q)
                            *reinterpret_cast<uint4 *>(pb + 8 * q) = make_uint4(wb[4 * q], wb[4 * q + 1], wb[4 * q + 2], wb[4 * q + 3]);
                    }
                } else {
                    for (int j = 0; j < CW && u0 + j < L.nout; ++j)
                        ob[j] = __ushort_as_bfloat16((unsigned short)((wb[j >> 1] >> (16 * (j & 1))) & 0xFFFFu));
                }
              } while (0);
              if (fine) {
                // the columns this CTA just wrote are the next half-step's TMA operand: order the generic-proxy
                // stores before the async-proxy reads, then tell the producer
                fence_proxy_async_global();
                __syncwarp();
                if (lane == 0) mbar_arrive(&sig[g]);
              }
            }
            }
            TC_TIME(tw2);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                uint64_t *tb = &tempty_bar[a];
                if (!leader)
                    mbar_arrive_cluster_addr(mapa_rank0(tb));
                else
                    mbar_arrive(tb);
            }
            if (p.persist && !fine) {
                fence_proxy_async_global();
                __syncwarp();
                if (lane == 0)
                    for (int g = 0; g < gpt; ++g) mbar_arrive(&sig[g]);
            }
            ++tl;
            if (++rot == TC_HALVES) rot = 0;
#ifdef ISB_TC_TIMING
            tm_wait += tw1 - tw0;
            tm_chunk += tw2 - tw1;
            tm_post += clock64() - tw2;
#endif
        };
        // The sampling warps walk their tiles with plain nested loops (the same sequence TcJobIter produces for the producer
        // and the issuer): the generic iterator cost them ~36 instructions and three spilled words per tile.
        {
            const int nst_loop = p.persist ? p.nsteps_seg : 1;
            const int stride = gridDim.x / p.cg;
            job.hs = 0;
            for (int step = 0; step < nst_loop; ++step) {
                job.k = p.k0 + step;
                for (int pass = 0; pass < (p.persist ? 2 : 1); ++pass) {
                    const int layer = p.persist ? 1 - pass : p.layer;
                    const int nt = p.L[layer].n_tiles;
                    const int first = p.persist ? 0 : blockIdx.x / p.cg;
                    const int last = p.persist ? nt : p.m_tiles * nt;
                    job.layer = layer;
                    for (int tile = first; tile < last; tile += p.persist ? 1 : stride) {
                        if (p.persist) {
                            job.m0 = blockIdx.x * p.rows_per_cta;
                            job.n_blk = tile;
                            job.hs_first = tile == 0;
                        } else {
                            job.m0 = (tile / nt) * (TC_BM * p.cg) + crank * TC_BM;
                            job.n_blk = tile % nt;
                            job.hs_first = false;
                        }
                        if (layer)
                            epi_tile(std::integral_constant<int, 1>{});
                        else
                            epi_tile(std::integral_constant<int, 0>{});
                    }
                }
            }
        }
#ifdef ISB_TC_TIMING
        if (lane == 0 && blockIdx.x < 296) {
            long long *o = g_tc_timing + ((size_t)blockIdx.x * 16 + (warp & 15)) * 4;
            o[0] = clock64() - tm_start; o[1] = tm_wait; o[2] = tm_chunk; o[3] = tm_post;
        }
#endif
    }
    tc_fence_before();
    cluster_sync_all();  // neither CTA frees its TMEM or retires while the pair's MMAs / remote arrives can be in flight
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

#ifdef ISB_TC_TIMING
extern "C" int isb_debug_tc_timing(long long *out, int n) {
    return (int)cudaMemcpyFromSymbol(out, g_tc_timing, sizeof(long long) * (size_t)std::min(n, 296 * 16 * 4));
}
#endif

__global__ void bias_to_float_kernel(const double *b, int n, int npad, float *o) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < npad) o[i] = i < n ? (float)b[i] : 0.f;
}
static int make_float_bias(isb_ctx *ctx, const double *d_b, int n, float **out) {
    const int npad = (n + 15) / 16 * 16;
    ISB_CUDA(ctx, cudaMalloc(out, (size_t)npad * sizeof(float)));
    bias_to_float_kernel<<<(npad + 255) / 256, 256, 0, ctx->stream>>>(d_b, n, npad, *out);
    ISB_CUDA(ctx, cudaGetLastError());
    ISB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return ISB_OK;
}

// bf16 / fp16 +-1 operand matrix -> canonical int8 spins (the sign bit is bit 15 in both formats)
__global__ void bf16_to_spins_kernel(const __nv_bfloat16 *b, int64_t ldb, int8_t *s, int64_t lds, int n, int R) {
    const int64_t total = (int64_t)R * n;
    for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = idx / n;
        const int u = (int)(idx % n);
        s[r * lds + u] = (__bfloat16_as_ushort(b[r * ldb + u]) & 0x8000u) ? (int8_t)-1 : (int8_t)1;
    }
}

// int8 +-1 -> +-1 operand matrix in bf16 (one = 0x3F80) or fp16 (one = 0x3C00), pad columns zero
__global__ void spins_to_bf16_kernel(const int8_t *s, int64_t lds, __nv_bfloat16 *o, int64_t ldo, int n, int R,
                                     unsigned short one) {
    const int64_t total = (int64_t)R * ldo;
    for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = idx / ldo;
        const int u = (int)(idx % ldo);
        unsigned short v = 0;
        if (u < n) v = s[r * lds + u] > 0 ? one : (unsigned short)(one | 0x8000u);
        o[idx] = __ushort_as_bfloat16(v);
    }
}

// ------------------------------------------------------------------ host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult qr;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qr) == cudaSuccess &&
            qr == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
    }
    return fn;
}

// 3-D bf16 operand [slabs][rows][ld] (cols valid per slab), box = {64 cols, 128 rows, 1 slab}: the A operand.
// An ordinary [R][K] spin matrix is the 1-slab case; row-sharded models keep the spins block-major [G][R][nb].
// esz = bytes per element: 2 (bf16 / fp16 terms) or 1 (int8 digit planes: box of 128 elements = the same 128 bytes)
static int make_map_a(isb_ctx *ctx, CUtensorMap *map, const void *base, int slabs, int rows, int cols, int64_t ld, int esz = 2) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) return fail(ctx, ISB_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
    cuuint64_t dims[3] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)slabs};
    cuuint64_t strides[2] = {(cuuint64_t)ld * esz, (cuuint64_t)ld * esz * (cuuint64_t)rows};
    cuuint32_t box[3] = {(cuuint32_t)(128 / esz), (cuuint32_t)TC_BM, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = fn(map, esz == 1 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void *>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS)
        return fail(ctx, ISB_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) for %d x %d x %d, ld %lld", (int)r, slabs, rows, cols, (long long)ld);
    return ISB_OK;
}

// 2-D bf16 matrix [rows][ld] (cols valid), box = {64 cols, box_rows}, 128B swizzle, OOB -> 0
static int make_map(isb_ctx *ctx, CUtensorMap *map, const void *base, int rows, int cols, int64_t ld, int box_rows, int esz = 2) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) return fail(ctx, ISB_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * esz};
    cuuint32_t box[2] = {(cuuint32_t)(128 / esz), (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, esz == 1 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void *>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(ctx, ISB_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) for %d x %d, ld %lld", (int)r, rows, cols, (long long)ld);
    return ISB_OK;
}

// fp16 term of x (round to nearest even) and its exact value
static unsigned short fp16_rne(double x, double *back) {
    const __half h = __double2half(x);
    *back = (double)__half2float(h);
    unsigned short bits;
    memcpy(&bits, &h, 2);
    return bits;
}

static unsigned short bf16_rne(double x, double *back) {
    float f = (float)x;
    uint32_t u;
    memcpy(&u, &f, 4);
    const uint32_t r = u + 0x7FFFu + ((u >> 16) & 1u);
    const unsigned short h = (unsigned short)(r >> 16);
    uint32_t ub = (uint32_t)h << 16;
    float fb;
    memcpy(&fb, &ub, 4);
    *back = (double)fb;
    return h;
}

// Tile width for a one-launch-per-half-step GEMM: the launch takes waves x bn "column units" of MMA time, so
// minimise ceil(m_tiles * ceil(nout / bn) / SMs) * bn over the legal widths (multiples of 16 up to 256).
static int pick_bn_waves(int nout, int m_tiles, int num_sms /* CTAs, or CTA pairs, that run tiles concurrently */, int bn_max = TC_BN_MAX) {
    int best = 0;
    long best_cost = 0;
    for (int bn = bn_max; bn >= 64; bn -= 16) {
        const long tiles = (long)m_tiles * ((nout + bn - 1) / bn);
        const long cost = ((tiles + num_sms - 1) / num_sms) * bn;
        if (best == 0 || cost < best_cost) {
            best = bn;
            best_cost = cost;
        }
    }
    return best;
}

static int pick_bn(int nout, int bn_max = TC_BN_MAX) {
    const int nt = (nout + bn_max - 1) / bn_max;
    int bn = ((nout + nt - 1) / nt + 15) / 16 * 16;
    return bn < 16 ? 16 : bn;
}

// Row pitch (elements) of a K-major bf16 operand with k valid columns.  A TMA box reads 128-256 rows at this pitch at
// once: a pitch that is a multiple of 1 KiB would put all of them on a few L2 slices, so such pitches get one more
// 128-byte line.
static int tc_pitch(int k, int esz = 2) {
    int ld = (k + 15) / 16 * 16;
    if ((ld * esz) % 1024 == 0) ld += 128 / esz;
    return ld;
}

// ---- int8 digit planes (ISB_PREC_I8X*)
// Fixed-point grid of P x 8 bits for couplings of magnitude <= amax: quantum q0 = 2^e (a power of two) such that every
// |W| / q0 rounds to an integer that P balanced base-256 digits (each in [-128, 127]; the top one in [-127, 127]) hold.
static long long i8_max_int(int P) {
    long long m = 0;
    for (int t = 0; t < P; ++t) m = m * 256 + 127;
    return m;
}
double i8_quantum(double amax, int P) {
    if (!(amax > 0.0)) return ldexp(1.0, -8 * P);
    int e;
    frexp(amax, &e);                       // amax = f 2^e, f in [0.5, 1)
    double q0 = ldexp(1.0, e - (8 * P - 1));  // amax / q0 < 2^(8P-1)
    if (rint(amax / q0) > (double)i8_max_int(P)) q0 *= 2.0;
    return q0;
}
// w (an integer, |w| <= i8_max_int(P)) -> P balanced digits, most significant first
__host__ __device__ inline void i8_digits(long long w, int P, int8_t *d) {
    for (int t = P - 1; t >= 0; --t) {
        long long r = ((w % 256) + 256) % 256;   // w mod 256 in [0, 255]
        if (r > 127) r -= 256;                    // balanced: [-128, 127]
        d[t] = (int8_t)r;
        w = (w - r) / 256;
    }
}
__host__ __device__ inline long long i8_quantize(double w, double q0, long long maxint) {
    double x = rint(w / q0);                      // q0 is a power of two: the division is exact
    if (x > (double)maxint) x = (double)maxint;
    if (x < -(double)maxint) x = -(double)maxint;
    return (long long)x;
}

static int prec_terms(int prec) {
    switch (prec) {
        case ISB_PREC_BF16X3: case ISB_PREC_I8X3: return 3;
        case ISB_PREC_BF16X2: case ISB_PREC_FP16X2: case ISB_PREC_I8X2: return 2;
        case ISB_PREC_I8X4: return 4;
        default: return 1;
    }
}
static bool prec_is_i8(int prec) { return prec == ISB_PREC_I8X2 || prec == ISB_PREC_I8X3 || prec == ISB_PREC_I8X4; }

// Units per tile of the stacked int8 layout (fixed when the model is built: it is part of the storage order).  The MMA
// takes N = P * bn <= 256 columns; a tile costs its N columns of tensor time plus a fixed part — the A tile is read once
// per K block whatever N is, the accumulator hand-over, and above all the per-tile code of the sampling warps (measured
// on config 4: 512 hidden units as 7 tiles of 80 beat 8 tiles of 64 by 3 % although they pad the layer to 560) — so
// minimise tiles x (N + 160) over the multiples of 16.
static int i8_pick_bn(int nout, int P) {
    int best = 16;
    long best_cost = 0;
    for (int bn = 16; bn * P <= TC_BN_MAX; bn += 16) {
        const long cost = (long)((nout + bn - 1) / bn) * (bn * P + 160);
        if (best_cost == 0 || cost <= best_cost) {
            best = bn;
            best_cost = cost;
        }
    }
    return best;
}
// row of (unit u, plane t) in the stacked matrix
__host__ __device__ inline int64_t i8_stack_row(int u, int t, int bn, int P) { return ((int64_t)(u / bn) * P + t) * bn + u % bn; }

// int8 digit planes of a bipartite model (host side): both orientations, the diagonal of a square model split off when
// it dominates the couplings (the pinning term of the MultiSpinFlip embedding)
static int bip_tc_model_init_i8(isb_model *m, TcModel *t, const double *W) {
    isb_ctx *ctx = m->ctx;
    const int nv = m->nv, nh = m->nh, P = t->P;
    double amax_off = 0.0, amax_diag = 0.0, amax_all = 0.0;
    for (int i = 0; i < nv; ++i)
        for (int j = 0; j < nh; ++j) {
            const double a = fabs(W[(size_t)i * nh + j]);
            amax_all = std::max(amax_all, a);
            if (nv == nh && i == j) amax_diag = std::max(amax_diag, a); else amax_off = std::max(amax_off, a);
        }
    const bool split = nv == nh && amax_diag > 2.0 * amax_off;
    t->q0 = i8_quantum(split ? amax_off : amax_all, P);
    const long long maxint = i8_max_int(P);
    t->ldkv = tc_pitch(nv, 1);
    t->ldkh = tc_pitch(nh, 1);
    t->bn_h = i8_pick_bn(nh, P);
    t->bn_v = i8_pick_bn(nv, P);
    // stacked storage: [tile][plane][unit in tile][K]; rows of the padding units of the last tile stay zero
    t->rows_t = (nh + t->bn_h - 1) / t->bn_h * t->bn_h * P; t->cols_t = nv;
    t->rows_n = (nv + t->bn_v - 1) / t->bn_v * t->bn_v * P; t->cols_n = nh;
    std::vector<int8_t> wt((size_t)t->rows_t * t->ldkv, 0), wn((size_t)t->rows_n * t->ldkh, 0);
    std::vector<double> dg;
    if (split) dg.assign((size_t)nv, 0.0);
    // L1 norms (in quanta) of the rows of both orientations: a contraction with +-1 spins cannot exceed them
    std::vector<long long> l1v((size_t)nv, 0), l1h((size_t)nh, 0);
    for (int i = 0; i < nv; ++i)
        for (int j = 0; j < nh; ++j) {
            const double w = W[(size_t)i * nh + j];
            if (split && i == j) {
                dg[i] = rint(w / t->q0) * t->q0;   // on the grid, not clamped: the epilogue adds it in float / double
                continue;
            }
            int8_t d[TC_PMAX];
            const long long wi = i8_quantize(w, t->q0, maxint);
            l1v[i] += wi < 0 ? -wi : wi;
            l1h[j] += wi < 0 ? -wi : wi;
            i8_digits(wi, P, d);
            for (int term = 0; term < P; ++term) {
                wt[(size_t)i8_stack_row(j, term, t->bn_h, P) * t->ldkv + i] = d[term];
                wn[(size_t)i8_stack_row(i, term, t->bn_v, P) * t->ldkh + j] = d[term];
            }
        }
    long long l1max = 0;
    for (long long v : l1v) l1max = std::max(l1max, v);
    for (long long v : l1h) l1max = std::max(l1max, v);
    t->i8_wide = l1max < (1ll << 31);
    ISB_CUDA(ctx, cudaMalloc(&t->Wt[0], wt.size()));
    ISB_CUDA(ctx, cudaMalloc(&t->Wn[0], wn.size()));
    ISB_CUDA(ctx, cudaMemcpy(t->Wt[0], wt.data(), wt.size(), cudaMemcpyHostToDevice));
    ISB_CUDA(ctx, cudaMemcpy(t->Wn[0], wn.data(), wn.size(), cudaMemcpyHostToDevice));
    if (split) {
        std::vector<float> dgf(((size_t)nv + 15) / 16 * 16, 0.f);
        for (int i = 0; i < nv; ++i) dgf[i] = (float)dg[i];
        ISB_CUDA(ctx, cudaMalloc(&t->diag_d, dg.size() * sizeof(double)));
        ISB_CUDA(ctx, cudaMalloc(&t->diag_f, dgf.size() * sizeof(float)));
        ISB_CUDA(ctx, cudaMemcpy(t->diag_d, dg.data(), dg.size() * sizeof(double), cudaMemcpyHostToDevice));
        ISB_CUDA(ctx, cudaMemcpy(t->diag_f, dgf.data(), dgf.size() * sizeof(float), cudaMemcpyHostToDevice));
    }
    return ISB_OK;
}

int bip_tc_model_init(isb_model *m, const double *W /*[nv][nh] row-major*/) {
    isb_ctx *ctx = m->ctx;
    TcModel *t = new TcModel();
    m->tc = t;
    t->P = prec_terms(m->prec);
    t->f16 = m->prec == ISB_PREC_FP16X2 || m->prec == ISB_PREC_FP16X1;
    t->i8 = prec_is_i8(m->prec);
    const int nv = m->nv, nh = m->nh;
    const int esz = t->i8 ? 1 : 2;
    if (t->i8) {
        int rc = bip_tc_model_init_i8(m, t, W);
        if (rc) return rc;
    } else {
    if (t->f16) {
        double amax = 0.0;
        for (size_t i = 0; i < (size_t)nv * nh; ++i) amax = std::max(amax, fabs(W[i]));
        if (amax > 0.0) {
            int e;
            frexp(amax, &e);                 // amax = f 2^e, f in [0.5, 1)
            t->wscale = ldexp(1.0, 14 - e);  // amax * wscale in [2^13, 2^14): far below fp16's 65504
        }
    }
    t->ldkv = tc_pitch(nv);
    t->ldkh = tc_pitch(nh);
    t->bn_h = pick_bn(nh);
    t->bn_v = pick_bn(nv);
    t->rows_t = nh; t->cols_t = nv; t->rows_n = nv; t->cols_n = nh;
    std::vector<unsigned short> wt((size_t)nh * t->ldkv), wn((size_t)nv * t->ldkh);
    std::vector<double> res((size_t)nv * nh);
    for (size_t i = 0; i < res.size(); ++i) res[i] = W[i] * t->wscale;  // a power of two: exact
    for (int term = 0; term < t->P; ++term) {
        std::fill(wt.begin(), wt.end(), 0);
        std::fill(wn.begin(), wn.end(), 0);
        for (int i = 0; i < nv; ++i)
            for (int j = 0; j < nh; ++j) {
                double back;
                const unsigned short hbits = t->f16 ? fp16_rne(res[(size_t)i * nh + j], &back) : bf16_rne(res[(size_t)i * nh + j], &back);
                res[(size_t)i * nh + j] -= back;
                wt[(size_t)j * t->ldkv + i] = hbits;
                wn[(size_t)i * t->ldkh + j] = hbits;
            }
        ISB_CUDA(ctx, cudaMalloc(&t->Wt[term], wt.size() * 2));
        ISB_CUDA(ctx, cudaMalloc(&t->Wn[term], wn.size() * 2));
        ISB_CUDA(ctx, cudaMemcpy(t->Wt[term], wt.data(), wt.size() * 2, cudaMemcpyHostToDevice));
        ISB_CUDA(ctx, cudaMemcpy(t->Wn[term], wn.data(), wn.size() * 2, cudaMemcpyHostToDevice));
    }
    }
    for (int term = 0; term < TC_PMAX; ++term) {
        const int src = (term < t->P && !t->i8) ? term : 0;
        const int sp = t->i8 ? t->P : 1;   // stacked planes: the box spans all planes of a tile
        int rc = make_map(ctx, &t->mapWt[term], t->Wt[src], t->rows_t, t->cols_t, t->ldkv, t->bn_h * sp, esz);
        if (rc) return rc;
        rc = make_map(ctx, &t->mapWn[term], t->Wn[src], t->rows_n, t->cols_n, t->ldkh, t->bn_v * sp, esz);
        if (rc) return rc;
    }
    int rc = make_float_bias(ctx, m->bb64, nh, &t->bias_hf);
    if (rc) return rc;
    return make_float_bias(ctx, m->hb64, nv, &t->bias_vf);
}

// The couplings exactly as the tensor path uses them (sum of the stored terms / digit planes, plus the split diagonal):
// Wout is [nv][nh] row-major (host).  Parity tests feed the oracle this matrix.
int bip_tc_effective_couplings(isb_model *m, double *Wout) {
    isb_ctx *ctx = m->ctx;
    TcModel *t = (TcModel *)m->tc;
    const int nv = m->nv, nh = m->nh;
    const size_t esz = t->i8 ? 1 : 2;
    std::vector<unsigned char> buf((size_t)t->rows_n * t->ldkh * esz);
    std::fill(Wout, Wout + (size_t)nv * nh, 0.0);
    for (int term = 0; term < t->P; ++term) {
        if (!t->i8 || term == 0)
            ISB_CUDA(ctx, cudaMemcpy(buf.data(), t->Wn[t->i8 ? 0 : term], buf.size(), cudaMemcpyDeviceToHost));
        const double wgt = t->i8 ? t->q0 * pow(256.0, t->P - 1 - term) : 1.0 / t->wscale;
        for (int i = 0; i < nv; ++i)
            for (int j = 0; j < nh; ++j) {
                const size_t k = (size_t)(t->i8 ? i8_stack_row(i, term, t->bn_v, t->P) : i) * t->ldkh + j;
                double v;
                if (t->i8) {
                    v = (double)reinterpret_cast<const int8_t *>(buf.data())[k];
                } else if (t->f16) {
                    __half hv;
                    memcpy(&hv, buf.data() + 2 * k, 2);
                    v = (double)__half2float(hv);
                } else {
                    const uint32_t ub = (uint32_t)reinterpret_cast<const unsigned short *>(buf.data())[k] << 16;
                    float fb;
                    memcpy(&fb, &ub, 4);
                    v = (double)fb;
                }
                Wout[(size_t)i * nh + j] += v * wgt;   // exact: every term is a multiple of the smallest term's ulp
            }
    }
    if (t->diag_d) {
        std::vector<double> dg((size_t)nv);
        ISB_CUDA(ctx, cudaMemcpy(dg.data(), t->diag_d, dg.size() * sizeof(double), cudaMemcpyDeviceToHost));
        for (int i = 0; i < nv; ++i) Wout[(size_t)i * nh + i] += dg[i];
    }
    return ISB_OK;
}

void bip_tc_model_free(isb_model *m) {
    TcModel *t = (TcModel *)m->tc;
    if (!t) return;
    for (int i = 0; i < TC_PMAX; ++i) {
        cudaFree(t->Wt[i]);
        cudaFree(t->Wn[i]);
    }
    cudaFree(t->bias_hf);
    cudaFree(t->bias_vf);
    cudaFree(t->diag_d);
    cudaFree(t->diag_f);
    delete t;
    m->tc = nullptr;
}

int bip_tc_ens_init(isb_ens *e) {
    isb_model *m = e->model;
    isb_ctx *ctx = m->ctx;
    TcModel *t = (TcModel *)m->tc;
    TcEns *s = new TcEns();
    e->tc = s;
    if (t->i8) {
        // int8 digit planes: the ensemble's canonical int8 spin arrays ARE the A operands (TMA zero-fills the columns
        // beyond nv / nh, whatever the pad bytes hold), and the epilogue writes +-1 bytes straight into them
        s->alias = true;
        s->Sv = reinterpret_cast<__nv_bfloat16 *>(e->spins);
        s->Sh = reinterpret_cast<__nv_bfloat16 *>(e->hidden);
        int rc = make_map_a(ctx, &s->mapSv, e->spins, 1, e->R, m->nv, e->lds, 1);
        if (rc) return rc;
        return make_map_a(ctx, &s->mapSh, e->hidden, 1, e->R, m->nh, e->ldh, 1);
    }
    ISB_CUDA(ctx, cudaMalloc(&s->Sv, (size_t)e->R * t->ldkv * 2));
    ISB_CUDA(ctx, cudaMalloc(&s->Sh, (size_t)e->R * t->ldkh * 2));
    int rc = make_map_a(ctx, &s->mapSv, s->Sv, 1, e->R, m->nv, t->ldkv);
    if (rc) return rc;
    return make_map_a(ctx, &s->mapSh, s->Sh, 1, e->R, m->nh, t->ldkh);
}

void bip_tc_ens_free(isb_ens *e) {
    TcEns *s = (TcEns *)e->tc;
    if (!s) return;
    if (!s->alias) {
        cudaFree(s->Sv);
        cudaFree(s->Sh);
    }
    delete s;
    e->tc = nullptr;
}

// Coupling tensor maps of orientation `orient` (1: Wt, hidden update; 0: Wn, visible update) whose box holds `bn`
// rows of W (half the tile width: each CTA of a pair loads half of the tile)
static int get_maps_b(isb_ctx *ctx, TcModel *t, int orient, int bn, CUtensorMap out[TC_PMAX]) {
    const int dflt = (orient == 1 ? t->bn_h : t->bn_v) * (t->i8 ? t->P : 1);
    const int esz = t->i8 ? 1 : 2;
    if (bn == dflt) {
        for (int i = 0; i < TC_PMAX; ++i) out[i] = orient == 1 ? t->mapWt[i] : t->mapWn[i];
        return ISB_OK;
    }
    for (auto &c : t->bn_cache)
        if (c.orient == orient && c.bn == bn) {
            for (int i = 0; i < TC_PMAX; ++i) out[i] = c.m[i];
            return ISB_OK;
        }
    TcModel::BnMaps c;
    c.orient = orient;
    c.bn = bn;
    for (int i = 0; i < TC_PMAX; ++i) {
        const int src = (i < t->P && !t->i8) ? i : 0;
        int rc = orient == 1 ? make_map(ctx, &c.m[i], t->Wt[src], t->rows_t, t->cols_t, t->ldkv, bn, esz)
                             : make_map(ctx, &c.m[i], t->Wn[src], t->rows_n, t->cols_n, t->ldkh, bn, esz);
        if (rc) return rc;
        out[i] = c.m[i];
    }
    t->bn_cache.push_back(c);
    return ISB_OK;
}

static void fill_layer(TcLayer &L, int nout, int kin, int bn, void *out_bf, int64_t ldo, const double *bias,
                       const float *bias_f, const double *F, uint32_t domain, int bk = TC_BK, int planes = 1) {
    L.nout = nout;
    L.kin = kin;
    L.bn = bn;
    L.bn_mma = bn * planes;
    L.n_tiles = (nout + bn - 1) / bn;
    L.num_kb = (kin + bk - 1) / bk;
    L.diag_f = nullptr;
    L.diag_d = nullptr;
    L.in_diag = nullptr;
    L.ld_in = 0;
    L.u_off = 0;
    L.kb_per_blk = L.num_kb;
    L.out_bf = out_bf;
    L.ldo = ldo;
    L.bias = bias;
    L.bias_f = bias_f;
    L.F = F;
    L.domain = domain;
    L.npeer = 0;
}

template <bool EXTF, int FMT>
static int launch_tc_inst(isb_ctx *ctx, const TcMaps &maps, const TcParams &p, int grid) {
    ISB_CUDA(ctx, cudaFuncSetAttribute(bip_tc_kernel<EXTF, FMT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TC_SMEM));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(TC_THREADS);
    cfg.dynamicSmemBytes = TC_SMEM;
    cfg.stream = ctx->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    ISB_CUDA(ctx, cudaLaunchKernelEx(&cfg, bip_tc_kernel<EXTF, FMT>, maps, p));
    return ISB_OK;
}

// grid = CTAs (even: CTA pairs)
static int launch_tc(isb_ctx *ctx, const TcMaps &maps, const TcParams &p, int grid, bool extf) {
    if (p.fmt == 2) return extf ? launch_tc_inst<true, 2>(ctx, maps, p, grid) : launch_tc_inst<false, 2>(ctx, maps, p, grid);
    if (p.fmt == 1) return extf ? launch_tc_inst<true, 1>(ctx, maps, p, grid) : launch_tc_inst<false, 1>(ctx, maps, p, grid);
    return extf ? launch_tc_inst<true, 0>(ctx, maps, p, grid) : launch_tc_inst<false, 0>(ctx, maps, p, grid);
}

// Steps [k0, k0 + nseg) of a run: one chain-resident launch when the replicas fill the SMs, else 2 * nseg
// half-step launches.
static int launch_steps(isb_ens *e, int rule, int fluct_mode, const double *d_Fv, const double *d_Fh, int64_t nsteps,
                        int64_t k0, int64_t nseg, const double *d_T, int64_t steps_per_T, uint64_t seed,
                        uint64_t step_offset) {
    isb_model *m = e->model;
    isb_ctx *ctx = m->ctx;
    TcModel *t = (TcModel *)m->tc;
    TcEns *s = (TcEns *)e->tc;
    const int m_tiles = (e->R + 2 * TC_BM - 1) / (2 * TC_BM);   // tiles of a CTA pair's 256 replicas
    const bool extf = fluct_mode != ISB_FLUCT_PHILOX;
    // chain-resident mode pays off when every SM gets a (nearly) full 128-row block of replicas to itself
    bool persist = (e->R + ctx->num_sms - 1) / ctx->num_sms >= 96;
    // ISB_TC_PERSIST=0|1 forces a launch mode (the tests run both on the same ensemble)
    if (const char *env = getenv("ISB_TC_PERSIST")) persist = atoi(env) != 0 && e->R >= 1;
    // tile widths: least padding per CTA in chain-resident mode, fewest (waves x width) otherwise
    // (int8 digit planes: the tile width is part of the stacked storage order, fixed when the model was built)
    const int sp = t->i8 ? t->P : 1;
    const int bn_h = (persist || t->i8) ? t->bn_h : pick_bn_waves(m->nh, m_tiles, ctx->num_sms / 2);
    const int bn_v = (persist || t->i8) ? t->bn_v : pick_bn_waves(m->nv, m_tiles, ctx->num_sms / 2);
    TcMaps maps;
    maps.A[1] = s->mapSv;
    maps.A[0] = s->mapSh;
    int rcm = get_maps_b(ctx, t, 1, bn_h * sp / 2, maps.B[1]);
    if (rcm) return rcm;
    rcm = get_maps_b(ctx, t, 0, bn_v * sp / 2, maps.B[0]);
    if (rcm) return rcm;
    TcParams p{};
    p.cg = 2;
    const int bk = t->i8 ? TC_BK8 : TC_BK;
    fill_layer(p.L[1], m->nh, m->nv, bn_h, s->Sh, t->i8 ? e->ldh : t->ldkh, m->bb64, t->bias_hf, d_Fh, DOM_BIP_HIDDEN, bk, sp);
    fill_layer(p.L[0], m->nv, m->nh, bn_v, s->Sv, t->i8 ? e->lds : t->ldkv, m->hb64, t->bias_vf, d_Fv, DOM_BIP_VISIBLE, bk, sp);
    if (t->diag_d) {  // square model with the diagonal split off: unit u's own input spin is column u of the input layer
        p.L[1].diag_f = p.L[0].diag_f = t->diag_f;
        p.L[1].diag_d = p.L[0].diag_d = t->diag_d;
        p.L[1].in_diag = e->spins;  p.L[1].ld_in = e->lds;
        p.L[0].in_diag = e->hidden; p.L[0].ld_in = e->ldh;
    }
    for (int term = 0; term < TC_PMAX; ++term) {
        p.i8_sd[term] = term < t->P ? t->q0 * pow(256.0, t->P - 1 - term) : 0.0;
        p.i8_sf[term] = (float)p.i8_sd[term];
    }
    // plane recombination of the fast sampling path (i8_field16): pairs are exact up to K = 65000, all three planes of
    // 24-bit couplings when the model's row L1 norms allow it
    p.i8_comb = std::max(m->nv, m->nh) <= 65000 ? ((t->P == 3 && t->i8_wide) ? 2 : 1) : 0;
    p.R = e->R;
    p.P = t->P;
    p.rule = rule;
    p.fluct_mode = fluct_mode;
    p.nsteps = nsteps;
    p.Tsched = d_T;
    p.tscale = e->d_tscale;
    p.steps_per_T = steps_per_T;
    p.seed = seed;
    p.keys = philox_keys(seed);
    p.fmt = t->i8 ? 2u : (t->f16 ? 1u : 0u);
    p.acc_scale = (float)(1.0 / t->wscale);
    p.m_tiles = m_tiles;
    for (int l = 0; l < 2; ++l) {
        p.sig_gpt[l] = (p.L[l].bn + TC_GW - 1) / TC_GW;
        if (p.L[l].n_tiles * p.sig_gpt[l] > TC_SIG_MAX) persist = false;  // more progress barriers than the CTA holds
    }
    if (persist) {
        p.persist = 1;
        p.sig_fine = 1;
        // A CTA's time per step does not depend on how many of its 128 tile rows hold replicas, and these runs are
        // POWER-capped (C4: ~1000 W, 1.75 GHz of 1.965): full tiles on fewer SMs do the same work per cycle with fewer
        // SMs drawing power — 16384 chains as 128 CTAs x 128 rows instead of 148 x 111 measured 0.313 -> 0.326 of the
        // bf16 burst rate at 1.84 GHz.
        p.rows_per_cta = TC_BM;
        p.nsteps_seg = (int)nseg;
        p.k0 = k0;
        p.step_abs0 = step_offset + (uint64_t)k0;
        const int grid = ((e->R + TC_BM - 1) / TC_BM + 1) / 2 * 2;  // an odd last CTA gets a peer without replicas
        int rc = launch_tc(ctx, maps, p, grid, extf);
        if (rc) return rc;
        e->last_launches += 1;
        return ISB_OK;
    }
    for (int64_t k = k0; k < k0 + nseg; ++k)
        for (int layer = 1; layer >= 0; --layer) {
            p.persist = 0;
            p.layer = layer;
            p.k0 = k;
            p.step_abs0 = step_offset + (uint64_t)k;
            const int grid = std::min(p.L[layer].n_tiles * p.m_tiles, ctx->num_sms / 2) * 2;
            int rc = launch_tc(ctx, maps, p, grid, extf);
            if (rc) return rc;
            e->last_launches += 1;
        }
    return ISB_OK;
}

// ------------------------------------------------------------------ row-sharded symmetric SCA (BASELINE config 5)
// Global problem: N spins, W = (J + qI)/2 symmetric (the MultiSpinFlip embedding, demo.jl:82-90), R replicas.
// Rank g of G owns the output units [g*nb, (g+1)*nb) of BOTH half-steps (W' = W), keeps W[block, :] as bf16
// split terms, and needs the full previous layer as the K operand: the spin matrices are kept block-major
// [G][R][nb] so that every rank's freshly sampled [R][nb] block is one contiguous all-gather contribution.

// Synthetic SK coupling J_ij = J_ji = g(min, max) / sqrt(N), g ~ N(0,1) by Box-Muller on two Philox words.
__device__ __forceinline__ double sk_coupling(uint64_t seed, int n, int i, int j) {
    if (i == j) return 0.0;
    const uint32_t a = (uint32_t)min(i, j), b = (uint32_t)max(i, j);
    const Philox4 w = philox4x32_10(a, b, 0u, 5u << 28, (uint32_t)seed, (uint32_t)(seed >> 32));
    const double u1 = ((double)w.x + 0.5) * 2.3283064365386962890625e-10;
    const double u2 = ((double)w.y + 0.5) * 2.3283064365386962890625e-10;
    return sqrt(-2.0 * log(u1)) * cospi(2.0 * u2) * rsqrt((double)n);
}
__device__ __forceinline__ unsigned short bf16_rne_dev(double x, double *back) {
    const float f = (float)x;
    const uint32_t u = __float_as_uint(f);
    const uint32_t r = u + 0x7FFFu + ((u >> 16) & 1u);
    const unsigned short h = (unsigned short)(r >> 16);
    *back = (double)__uint_as_float((uint32_t)h << 16);
    return h;
}
// Fills the P bf16 split terms of W[row0 + r][c] = (J + qI)/2 (generated, or taken from Wrows when given).
__global__ void shard_fill_kernel(int n, int row0, int nrows, uint64_t seed, double q, const double *Wrows, int P,
                                  __nv_bfloat16 *t0, __nv_bfloat16 *t1, __nv_bfloat16 *t2) {
    const int64_t total = (int64_t)nrows * n;
    for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
        const int r = (int)(idx / n), c = (int)(idx % n);
        double w = Wrows ? Wrows[idx] : 0.5 * (sk_coupling(seed, n, row0 + r, c) + (row0 + r == c ? q : 0.0));
        double back;
        t0[idx] = __ushort_as_bfloat16(bf16_rne_dev(w, &back));
        if (P > 1) {
            w -= back;
            t1[idx] = __ushort_as_bfloat16(bf16_rne_dev(w, &back));
        }
        if (P > 2) {
            w -= back;
            t2[idx] = __ushort_as_bfloat16(bf16_rne_dev(w, &back));
        }
    }
}
// int8 digit planes of the same rows: off-diagonal couplings on the grid q0, the diagonal kept apart (on the grid too)
__global__ void shard_fill_i8_kernel(int n, int row0, int nrows, uint64_t seed, double q, const double *Wrows, int P,
                                     double q0, long long maxint, int8_t *stack, int bn, double *diag_d, float *diag_f) {
    const int64_t total = (int64_t)nrows * n;
    for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
        const int r = (int)(idx / n), c = (int)(idx % n);
        const double w = Wrows ? Wrows[idx] : 0.5 * (sk_coupling(seed, n, row0 + r, c) + (row0 + r == c ? q : 0.0));
        int8_t d[TC_PMAX] = {0, 0, 0, 0};
        if (row0 + r == c) {
            const double dg = rint(w / q0) * q0;
            diag_d[r] = dg;
            diag_f[r] = (float)dg;
        } else {
            i8_digits(i8_quantize(w, q0, maxint), P, d);
        }
        for (int t = 0; t < P; ++t) stack[i8_stack_row(r, t, bn, P) * n + c] = d[t];   // [tile][plane][unit][K]
    }
}
__global__ void sk_rows_kernel(int n, uint64_t seed, int row0, int nrows, double *out) {
    const int64_t total = (int64_t)nrows * n;
    for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x)
        out[idx] = sk_coupling(seed, n, row0 + (int)(idx / n), (int)(idx % n));
}

int sk_rows_device(isb_ctx *ctx, int n, uint64_t seed, int row0, int nrows, double *d_out) {
    sk_rows_kernel<<<ctx->num_sms * 8, 256, 0, ctx->stream>>>(n, seed, row0, nrows, d_out);
    ISB_CUDA(ctx, cudaGetLastError());
    return ISB_OK;
}

int shard_model_init(isb_model *m, const double *Wrows, uint64_t seed, double q, double wmax) {
    isb_ctx *ctx = m->ctx;
    TcModel *t = new TcModel();
    m->tc = t;
    t->P = prec_terms(m->prec);
    t->i8 = prec_is_i8(m->prec);
    const int esz = t->i8 ? 1 : 2;
    const int n = m->nv, nb = m->shard_nb;
    t->ldkv = t->ldkh = n;
    t->bn_h = t->bn_v = t->i8 ? i8_pick_bn(nb, t->P) : pick_bn(nb);
    t->rows_t = t->rows_n = t->i8 ? (nb + t->bn_h - 1) / t->bn_h * t->bn_h * t->P : nb;
    t->cols_t = t->cols_n = n;
    const size_t elems = (size_t)nb * n;
    double *dW = nullptr;
    if (Wrows) {
        ISB_CUDA(ctx, cudaMalloc(&dW, elems * sizeof(double)));
        ISB_CUDA(ctx, cudaMemcpyAsync(dW, Wrows, elems * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    }
    if (t->i8) {
        ISB_CUDA(ctx, cudaMalloc(&t->Wt[0], (size_t)t->rows_t * n));
        ISB_CUDA(ctx, cudaMemsetAsync(t->Wt[0], 0, (size_t)t->rows_t * n, ctx->stream));
    } else {
        for (int term = 0; term < t->P; ++term) ISB_CUDA(ctx, cudaMalloc(&t->Wt[term], elems * esz));
    }
    if (t->i8) {
        // The grid must be the same on every rank (the trajectory may not depend on the sharding): the caller passes
        // the largest off-diagonal |W| of the WHOLE matrix (wmax); for the synthetic instance it is bounded a priori:
        // |J_ij| = |g| / sqrt(n) with |g| <= sqrt(-2 ln 2^-33) < 6.77 (Box-Muller on a 32-bit uniform), W = J / 2.
        if (!Wrows) wmax = 0.5 * 6.77 / sqrt((double)n);
        if (!(wmax > 0.0) && Wrows) {   // not given: this block's own maximum (single-block models)
            for (int r = 0; r < nb; ++r)
                for (int c = 0; c < n; ++c)
                    if (m->shard_g * nb + r != c) wmax = std::max(wmax, fabs(Wrows[(size_t)r * n + c]));
        }
        t->q0 = i8_quantum(wmax, t->P);
        ISB_CUDA(ctx, cudaMalloc(&t->diag_d, (size_t)nb * sizeof(double)));
        ISB_CUDA(ctx, cudaMalloc(&t->diag_f, (size_t)nb * sizeof(float)));
        shard_fill_i8_kernel<<<ctx->num_sms * 8, 256, 0, ctx->stream>>>(
            n, m->shard_g * nb, nb, seed, q, dW, t->P, t->q0, i8_max_int(t->P), (int8_t *)t->Wt[0], t->bn_h, t->diag_d, t->diag_f);
    } else {
        shard_fill_kernel<<<ctx->num_sms * 8, 256, 0, ctx->stream>>>(n, m->shard_g * nb, nb, seed, q, dW, t->P, t->Wt[0],
                                                                     t->Wt[1], t->Wt[2]);
    }
    ISB_CUDA(ctx, cudaGetLastError());
    ISB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (dW) cudaFree(dW);
    for (int term = 0; term < TC_PMAX; ++term) {
        const int src = (term < t->P && !t->i8) ? term : 0;
        int rc = make_map(ctx, &t->mapWt[term], t->Wt[src], t->rows_t, n, n, t->bn_h * (t->i8 ? t->P : 1), esz);
        if (rc) return rc;
    }
    int rc = make_float_bias(ctx, m->bb64, nb, &t->bias_hf);
    if (rc) return rc;
    return make_float_bias(ctx, m->hb64, nb, &t->bias_vf);
}

int shard_elem_size(const isb_model *m) { return ((const TcModel *)m->tc)->i8 ? 1 : 2; }

int shard_halfstep_device(isb_model *m, int R, int replica_offset, int layer, int rule, const void *in_full, void *out_block,
                          int n_peers, void *const *peer_blocks, uint64_t seed, uint64_t step_abs, double T) {
    isb_ctx *ctx = m->ctx;
    TcModel *t = (TcModel *)m->tc;
    TcMaps maps;
    const int esz = t->i8 ? 1 : 2, bk = t->i8 ? TC_BK8 : TC_BK;
    int rc = make_map_a(ctx, &maps.A[layer], in_full, m->shard_G, R, m->shard_nb, m->shard_nb, esz);
    if (rc) return rc;
    maps.A[1 - layer] = maps.A[layer];
    const int m_tiles = (R + 2 * TC_BM - 1) / (2 * TC_BM);
    const int sp = t->i8 ? t->P : 1;   // int8: the tile width is part of the stacked storage order
    const int bn = t->i8 ? t->bn_h : pick_bn_waves(m->shard_nb, m_tiles, ctx->num_sms / 2);
    rc = get_maps_b(ctx, t, 1, bn * sp / 2, maps.B[1]);  // W is symmetric: one orientation serves both half-steps
    if (rc) return rc;
    for (int i = 0; i < TC_PMAX; ++i) maps.B[0][i] = maps.B[1][i];
    TcParams p{};
    fill_layer(p.L[layer], m->shard_nb, m->nv, bn, out_block, m->shard_nb,
               layer == 1 ? m->bb64 : m->hb64, layer == 1 ? t->bias_hf : t->bias_vf, nullptr,
               layer == 1 ? DOM_BIP_HIDDEN : DOM_BIP_VISIBLE, bk, sp);
    p.L[layer].u_off = m->shard_g * m->shard_nb;
    p.L[layer].num_kb = m->nv / bk;
    p.L[layer].kb_per_blk = m->shard_nb / bk;
    p.L[layer].npeer = n_peers;
    for (int q = 0; q < n_peers; ++q) p.L[layer].peer[q] = peer_blocks[q];
    if (t->i8) {  // the diagonal of W: unit u's own input spin sits in this rank's slab of the gathered input layer
        p.L[layer].diag_f = t->diag_f;
        p.L[layer].diag_d = t->diag_d;
        p.L[layer].in_diag = reinterpret_cast<const int8_t *>(in_full) + (size_t)m->shard_g * R * m->shard_nb;
        p.L[layer].ld_in = m->shard_nb;
    }
    for (int term = 0; term < TC_PMAX; ++term) {
        p.i8_sd[term] = term < t->P ? t->q0 * pow(256.0, t->P - 1 - term) : 0.0;
        p.i8_sf[term] = (float)p.i8_sd[term];
    }
    p.i8_comb = (int64_t)m->shard_nb * m->shard_G <= 65000 ? 1 : 0;   // (row L1 norms of generated rows are not known here: no all-int32 form)
    p.L[1 - layer] = p.L[layer];
    p.R = R;
    p.r_off = replica_offset;
    p.P = t->P;
    p.rule = rule;
    p.fluct_mode = ISB_FLUCT_PHILOX;
    p.Tsched = nullptr;
    p.fmt = t->i8 ? 2u : 0u;  // row-sharded models: bf16 terms or int8 digit planes
    p.acc_scale = 1.0f;
    p.T_direct = T;
    p.steps_per_T = 1;
    p.seed = seed;
    p.keys = philox_keys(seed);
    p.step_abs0 = step_abs;
    p.persist = 0;
    p.layer = layer;
    p.cg = 2;
    p.m_tiles = m_tiles;
    const int grid = std::min(p.L[layer].n_tiles * p.m_tiles, ctx->num_sms / 2) * 2;
    return launch_tc(ctx, maps, p, grid, false);
}

int bip_run_tc_device(isb_ens *e, int rule, int64_t nsteps, int fluct_mode, const double *d_Fv, const double *d_Fh,
                      uint64_t seed, uint64_t step_offset, const double *d_T, int64_t steps_per_T, int64_t trace_every,
                      double *d_E, int8_t *d_Sv, int8_t *d_Sh) {
    isb_model *m = e->model;
    isb_ctx *ctx = m->ctx;
    TcModel *t = (TcModel *)m->tc;
    TcEns *s = (TcEns *)e->tc;
    // the canonical int8 visible layer is the input of the first half-step; the hidden bf16 matrix is
    // produced by it (MomentumAnnealing reads the hidden layer's previous value from the int8 array)
    // (int8 digit planes: the canonical int8 arrays are the operands themselves — nothing to convert)
    const unsigned short one = t->f16 ? 0x3C00 : 0x3F80;
    if (!t->i8) {
        spins_to_bf16_kernel<<<ctx->num_sms * 4, 256, 0, ctx->stream>>>(e->spins, e->lds, s->Sv, t->ldkv, m->nv, e->R, one);
        spins_to_bf16_kernel<<<ctx->num_sms * 4, 256, 0, ctx->stream>>>(e->hidden, e->ldh, s->Sh, t->ldkh, m->nh, e->R, one);
        ISB_CUDA(ctx, cudaGetLastError());
        e->last_launches += 2;
    }
    auto sync_canonical = [&]() -> int {  // bf16 operand matrices -> the ensemble's int8 spins
        if (t->i8) return ISB_OK;
        bf16_to_spins_kernel<<<ctx->num_sms * 4, 256, 0, ctx->stream>>>(s->Sv, t->ldkv, e->spins, e->lds, m->nv, e->R);
        bf16_to_spins_kernel<<<ctx->num_sms * 4, 256, 0, ctx->stream>>>(s->Sh, t->ldkh, e->hidden, e->ldh, m->nh, e->R);
        ISB_CUDA(ctx, cudaGetLastError());
        e->last_launches += 2;
        return ISB_OK;
    };
    int64_t ntr = 0;
    const bool tracing = (d_E || d_Sv || d_Sh) && trace_every > 0;
    bool canonical_fresh = false;  // the int8 spins already hold the state of the last executed step
    for (int64_t k0 = 0; k0 < nsteps;) {
        const int64_t nseg = tracing ? std::min<int64_t>(trace_every - (k0 % trace_every), nsteps - k0)
                                     : std::min<int64_t>(nsteps - k0, 1 << 20);
        int rc = launch_steps(e, rule, fluct_mode, d_Fv, d_Fh, nsteps, k0, nseg, d_T, steps_per_T, seed, step_offset);
        if (rc) return rc;
        k0 += nseg;
        canonical_fresh = false;
        if (tracing && k0 % trace_every == 0) {
            rc = sync_canonical();
            if (rc) return rc;
            canonical_fresh = true;
            if (d_E) {
                rc = bip_energy_device(e, d_E + ntr * e->R);
                if (rc) return rc;
                e->last_launches += 2;
            }
            rc = bip_snapshot(e, ntr, d_Sv, d_Sh);
            if (rc) return rc;
            ++ntr;
        }
    }
    return canonical_fresh ? ISB_OK : sync_canonical();
}

}  // namespace isb
