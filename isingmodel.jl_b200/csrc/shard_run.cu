// shard_run.cu — the step loop of the row-sharded synchronous SCA (BASELINE config 5) behind the C ABI.
//
// isb_shard_halfstep_dev is one half-step of one rank's block; the loop around it — two replica groups, the exchange of
// the freshly sampled blocks after every half-step (the path's one real collective, north_star: "an all-gather of the
// spin vector each synchronous step"), the ordering between them — used to live in the Python host layer on torch.
// isb_shard_run_* is that loop inside the library, so that a C or Julia caller needs neither torch nor Python:
//   * the gathered spin matrices ([G][Rg][nb] per layer and replica group, +-1 in the operand format) and this rank's
//     blocks are owned here (cudaMalloc);
//   * exchange ISB_EXCH_NCCL: ncclAllGather on a side stream (libnccl.so.2 is resolved with dlopen when first needed,
//     the library does not link against it); the communicator is the caller's (isb_shard_run_set_nccl_comm) or created
//     from a unique id (isb_nccl_unique_id + isb_shard_run_init_nccl);
//   * exchange ISB_EXCH_COPY: every rank PUSHES its block into all ranks' gathered matrices with the copy engines
//     (peer pointers from CUDA IPC handles the caller passes around: isb_shard_run_ipc_export / _import), then signals
//     the peers and waits for theirs with stream memory operations (cuStreamWriteValue64 / cuStreamWaitValue64 on
//     IPC-mapped flag words) — no kernel spins, no SM is taken from the contraction;
//   * either way the replicas are split into two groups and one group's exchange runs on the side stream under the
//     other group's contraction (chains are independent).  ISB_EXCH_LOCAL: a single rank, no exchange.
// The noise is indexed by global (replica, step, unit): the trajectory is identical for every G and exchange.
#include <cuda.h>
#include <dlfcn.h>
#include <nccl.h>
#include <string.h>

#include <algorithm>
#include <cmath>
#include <vector>

#include "common.cuh"
#include "handles.hpp"

namespace isb {

// ---- libnccl through dlopen
struct NcclApi {
    void *lib = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
};
static NcclApi *nccl_api() {
    static NcclApi api;
    static bool tried = false;
    if (!tried) {
        tried = true;
        const char *names[] = {"libnccl.so.2", "libnccl.so"};
        for (const char *nm : names) {
            api.lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
            if (api.lib) break;
        }
        if (api.lib) {
            api.GetUniqueId = (decltype(api.GetUniqueId))dlsym(api.lib, "ncclGetUniqueId");
            api.CommInitRank = (decltype(api.CommInitRank))dlsym(api.lib, "ncclCommInitRank");
            api.CommDestroy = (decltype(api.CommDestroy))dlsym(api.lib, "ncclCommDestroy");
            api.AllGather = (decltype(api.AllGather))dlsym(api.lib, "ncclAllGather");
            api.GetErrorString = (decltype(api.GetErrorString))dlsym(api.lib, "ncclGetErrorString");
            if (!api.GetUniqueId || !api.CommInitRank || !api.CommDestroy || !api.AllGather || !api.GetErrorString) {
                dlclose(api.lib);
                api.lib = nullptr;
            }
        }
    }
    return api.lib ? &api : nullptr;
}

// Stream memory operations of the driver API, resolved at run time (the library must load on a box without a driver:
// it does not link against libcuda)
typedef CUresult (*StreamValue64Fn)(CUstream, CUdeviceptr, cuuint64_t, unsigned int);
static StreamValue64Fn driver_fn(const char *name) {
    void *p = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint(name, &p, cudaEnableDefault, &qr) == cudaSuccess && qr == cudaDriverEntryPointSuccess)
        return (StreamValue64Fn)p;
    return nullptr;
}
static CUresult stream_write64(cudaStream_t st, void *addr, uint64_t v) {
    static StreamValue64Fn fn = driver_fn("cuStreamWriteValue64");
    return fn ? fn((CUstream)st, (CUdeviceptr)addr, v, CU_STREAM_WRITE_VALUE_DEFAULT) : CUDA_ERROR_NOT_SUPPORTED;
}
static CUresult stream_wait_geq64(cudaStream_t st, void *addr, uint64_t v) {
    static StreamValue64Fn fn = driver_fn("cuStreamWaitValue64");
    return fn ? fn((CUstream)st, (CUdeviceptr)addr, v, CU_STREAM_WAIT_VALUE_GEQ) : CUDA_ERROR_NOT_SUPPORTED;
}

// [R][ld] int8 +-1 (host order) <-> block-major [G][Rg][nb] in the operand format, for the replicas [r0, r0 + Rg)
__global__ void shard_scatter_kernel(const int8_t *S, int64_t ld, int r0, int Rg, int G, int nb, int esz, void *full) {
    const int64_t total = (int64_t)G * Rg * nb;
    for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
        const int u = (int)(idx % nb);
        const int64_t t = idx / nb;
        const int rr = (int)(t % Rg), g = (int)(t / Rg);
        const bool up = S[(int64_t)(r0 + rr) * ld + (int64_t)g * nb + u] > 0;
        if (esz == 1)
            reinterpret_cast<int8_t *>(full)[idx] = up ? (int8_t)1 : (int8_t)-1;
        else
            reinterpret_cast<unsigned short *>(full)[idx] = up ? (unsigned short)0x3F80 : (unsigned short)0xBF80;
    }
}
__global__ void shard_collect_kernel(const void *full, int r0, int Rg, int G, int nb, int esz, int8_t *S, int64_t ld) {
    const int64_t total = (int64_t)G * Rg * nb;
    for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
        const int u = (int)(idx % nb);
        const int64_t t = idx / nb;
        const int rr = (int)(t % Rg), g = (int)(t / Rg);
        const bool neg = esz == 1 ? reinterpret_cast<const int8_t *>(full)[idx] < 0
                                  : (reinterpret_cast<const unsigned short *>(full)[idx] & 0x8000u) != 0;
        S[(int64_t)(r0 + rr) * ld + (int64_t)g * nb + u] = neg ? (int8_t)-1 : (int8_t)1;
    }
}

}  // namespace isb

using isb::fail;

#define ISB_TRY(expr)                  \
    do {                               \
        int _rc = (expr);              \
        if (_rc != ISB_OK) return _rc; \
    } while (0)

enum { SR_MAX_GROUPS = 2, SR_MAX_RANKS = 64 };

struct SrGroup {
    int r0 = 0, R = 0;
    void *full[2] = {nullptr, nullptr};   // gathered layer: [0] visible, [1] hidden; [G][R][nb]
    void *blk[2] = {nullptr, nullptr};    // this rank's freshly sampled block of each layer: [R][nb]
    cudaEvent_t ready[2] = {nullptr, nullptr};   // gathered layer complete (recorded on the exchange stream)
    bool pending[2] = {false, false};
    cudaEvent_t sampled = nullptr;               // half-step kernel done (recorded on the compute stream)
};

struct isb_shard_run {
    isb_model *model = nullptr;
    int R = 0, exchange = 0, G = 1, g = 0, nb = 0, n = 0, esz = 2, ngroups = 1;
    SrGroup grp[SR_MAX_GROUPS];
    cudaStream_t xstream = nullptr;
    // NCCL
    ncclComm_t comm = nullptr;
    bool own_comm = false;
    // copy-engine exchange: one allocation holds everything a peer must reach (the gathered matrices and the flag words)
    unsigned char *arena = nullptr;
    size_t arena_bytes = 0;
    size_t off_full[SR_MAX_GROUPS][2] = {}, off_flags = 0;
    unsigned char *peer_arena[SR_MAX_RANKS] = {};   // IPC-mapped arenas of the other ranks ([g] = own)
    bool peer_open[SR_MAX_RANKS] = {};
    uint64_t epoch[SR_MAX_GROUPS][2] = {};          // exchanges completed per (group, layer)
    uint64_t bar_epoch = 0;
    uint64_t *stage = nullptr;                      // [SR_MAX_GROUPS * 2 + 1] local words the signals are copied from
    int8_t *hostfmt = nullptr;                      // [R][n] int8 staging of set_spins / get_spins
    int64_t launches = 0;
    double last_ms = 0.0;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
};

// flag word of (source rank q, group, layer) in an arena; the last G words are the barrier flags
static size_t sr_flag_off(const isb_shard_run *s, int q, int gi, int layer) {
    return s->off_flags + ((size_t)(gi * 2 + layer) * s->G + q) * sizeof(uint64_t);
}
static size_t sr_bar_off(const isb_shard_run *s, int q) {
    return s->off_flags + ((size_t)SR_MAX_GROUPS * 2 * s->G + q) * sizeof(uint64_t);
}

extern "C" {

int isb_nccl_unique_id(void *id128) {
    if (!id128) return ISB_ERR_ARG;
    isb::NcclApi *api = isb::nccl_api();
    if (!api) return fail(nullptr, ISB_ERR_NCCL, "isb_nccl_unique_id: libnccl.so.2 could not be loaded");
    ncclUniqueId id;
    const ncclResult_t r = api->GetUniqueId(&id);
    if (r != ncclSuccess) return fail(nullptr, ISB_ERR_NCCL, "ncclGetUniqueId: %s", api->GetErrorString(r));
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    memcpy(id128, &id, 128);
    return ISB_OK;
}

int isb_shard_run_create(isb_model *m, int R, int exchange, isb_shard_run **out) {
    if (!m) return ISB_ERR_ARG;
    isb_ctx *ctx = m->ctx;
    ISB_LOCK(ctx);
    if (!out) return fail(ctx, ISB_ERR_ARG, "isb_shard_run_create: out is NULL");
    *out = nullptr;
    if (m->kind != ISB_KIND_SHARD) return fail(ctx, ISB_ERR_STATE, "isb_shard_run_create: not a row-sharded model");
    if (R <= 0) return fail(ctx, ISB_ERR_SIZE, "isb_shard_run_create: R = %d must be positive", R);
    if (exchange < ISB_EXCH_LOCAL || exchange > ISB_EXCH_COPY) return fail(ctx, ISB_ERR_ARG, "isb_shard_run_create: unknown exchange %d", exchange);
    if (m->shard_G > SR_MAX_RANKS) return fail(ctx, ISB_ERR_UNSUPPORTED, "isb_shard_run_create: more than %d blocks", SR_MAX_RANKS);
    if (exchange == ISB_EXCH_LOCAL && m->shard_G != 1)
        return fail(ctx, ISB_ERR_STATE, "isb_shard_run_create: ISB_EXCH_LOCAL needs a single block (this model is block %d of %d)", m->shard_g, m->shard_G);
    ISB_CUDA(ctx, cudaSetDevice(ctx->device));
    isb_shard_run *s = new isb_shard_run();
    s->model = m;
    m->refs.fetch_add(1);
    s->R = R;
    s->exchange = exchange;
    s->G = m->shard_G;
    s->g = m->shard_g;
    s->nb = m->shard_nb;
    s->n = m->nv;
    s->esz = isb::shard_elem_size(m);
    // two replica groups (whole 128-replica tiles in the first) when there is an exchange to hide and enough replicas
    s->ngroups = (exchange != ISB_EXCH_LOCAL && R >= 256) ? 2 : 1;
    const int half = s->ngroups == 2 ? (R / 2 + 127) / 128 * 128 : R;
    s->grp[0].r0 = 0;
    s->grp[0].R = half;
    s->grp[1].r0 = half;
    s->grp[1].R = R - half;
    if (s->grp[1].R <= 0) s->ngroups = 1;
    // arena: gathered matrices of every (group, layer), 256-byte aligned, then the flag words
    size_t off = 0;
    for (int gi = 0; gi < s->ngroups; ++gi)
        for (int l = 0; l < 2; ++l) {
            s->off_full[gi][l] = off;
            off += ((size_t)s->G * s->grp[gi].R * s->nb * s->esz + 255) / 256 * 256;
        }
    s->off_flags = off;
    off += ((size_t)SR_MAX_GROUPS * 2 + 1) * s->G * sizeof(uint64_t);
    s->arena_bytes = (off + 255) / 256 * 256;
    cudaError_t ce = cudaMalloc(&s->arena, s->arena_bytes);
    if (ce == cudaSuccess) ce = cudaMemset(s->arena, 0, s->arena_bytes);
    for (int gi = 0; gi < s->ngroups && ce == cudaSuccess; ++gi) {
        SrGroup &gr = s->grp[gi];
        for (int l = 0; l < 2 && ce == cudaSuccess; ++l) {
            gr.full[l] = s->arena + s->off_full[gi][l];
            ce = cudaMalloc(&gr.blk[l], (size_t)gr.R * s->nb * s->esz);
            if (ce == cudaSuccess) ce = cudaEventCreateWithFlags(&gr.ready[l], cudaEventDisableTiming);
        }
        if (ce == cudaSuccess) ce = cudaEventCreateWithFlags(&gr.sampled, cudaEventDisableTiming);
    }
    if (ce == cudaSuccess) ce = cudaMalloc(&s->hostfmt, (size_t)R * s->n);
    if (ce == cudaSuccess) ce = cudaMalloc(&s->stage, (SR_MAX_GROUPS * 2 + 1) * sizeof(uint64_t));
    if (ce == cudaSuccess) ce = cudaMemset(s->stage, 0, (SR_MAX_GROUPS * 2 + 1) * sizeof(uint64_t));
    if (ce == cudaSuccess) ce = cudaStreamCreateWithFlags(&s->xstream, cudaStreamNonBlocking);
    if (ce == cudaSuccess) ce = cudaEventCreate(&s->ev0);
    if (ce == cudaSuccess) ce = cudaEventCreate(&s->ev1);
    if (ce != cudaSuccess) {
        isb_shard_run_destroy(s);
        return fail(ctx, ISB_ERR_CUDA, "isb_shard_run_create: %s", cudaGetErrorString(ce));
    }
    s->peer_arena[s->g] = s->arena;
    *out = s;
    return ISB_OK;
}

void isb_shard_run_destroy(isb_shard_run *s) {
    if (!s) return;
    isb_model *m = s->model;
    {
        ISB_LOCK(m->ctx);
        cudaSetDevice(m->ctx->device);
        cudaStreamSynchronize(m->ctx->stream);
        if (s->xstream) cudaStreamSynchronize(s->xstream);
        if (s->own_comm && s->comm && isb::nccl_api()) isb::nccl_api()->CommDestroy(s->comm);
        for (int q = 0; q < s->G && q < SR_MAX_RANKS; ++q)
            if (s->peer_open[q]) cudaIpcCloseMemHandle(s->peer_arena[q]);
        for (int gi = 0; gi < SR_MAX_GROUPS; ++gi) {
            SrGroup &gr = s->grp[gi];
            for (int l = 0; l < 2; ++l) {
                cudaFree(gr.blk[l]);
                if (gr.ready[l]) cudaEventDestroy(gr.ready[l]);
            }
            if (gr.sampled) cudaEventDestroy(gr.sampled);
        }
        cudaFree(s->arena);
        cudaFree(s->stage);
        cudaFree(s->hostfmt);
        if (s->xstream) cudaStreamDestroy(s->xstream);
        if (s->ev0) cudaEventDestroy(s->ev0);
        if (s->ev1) cudaEventDestroy(s->ev1);
        delete s;
    }
    isb_model_destroy(m);
}

int isb_shard_run_set_nccl_comm(isb_shard_run *s, void *nccl_comm) {
    if (!s) return ISB_ERR_ARG;
    isb_ctx *ctx = s->model->ctx;
    ISB_LOCK(ctx);
    if (!nccl_comm) return fail(ctx, ISB_ERR_ARG, "isb_shard_run_set_nccl_comm: communicator is NULL");
    if (!isb::nccl_api()) return fail(ctx, ISB_ERR_NCCL, "isb_shard_run_set_nccl_comm: libnccl.so.2 could not be loaded");
    s->comm = (ncclComm_t)nccl_comm;
    s->own_comm = false;
    return ISB_OK;
}

int isb_shard_run_init_nccl(isb_shard_run *s, const void *id128) {
    if (!s) return ISB_ERR_ARG;
    isb_ctx *ctx = s->model->ctx;
    ISB_LOCK(ctx);
    if (!id128) return fail(ctx, ISB_ERR_ARG, "isb_shard_run_init_nccl: id is NULL");
    isb::NcclApi *api = isb::nccl_api();
    if (!api) return fail(ctx, ISB_ERR_NCCL, "isb_shard_run_init_nccl: libnccl.so.2 could not be loaded");
    ISB_CUDA(ctx, cudaSetDevice(ctx->device));
    ncclUniqueId id;
    memcpy(&id, id128, 128);
    const ncclResult_t r = api->CommInitRank(&s->comm, s->G, id, s->g);
    if (r != ncclSuccess) return fail(ctx, ISB_ERR_NCCL, "ncclCommInitRank (rank %d of %d): %s", s->g, s->G, api->GetErrorString(r));
    s->own_comm = true;
    return ISB_OK;
}

int isb_shard_run_ipc_export(isb_shard_run *s, void *handle64) {
    if (!s) return ISB_ERR_ARG;
    isb_ctx *ctx = s->model->ctx;
    ISB_LOCK(ctx);
    if (!handle64) return fail(ctx, ISB_ERR_ARG, "isb_shard_run_ipc_export: handle is NULL");
    ISB_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t h;
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    ISB_CUDA(ctx, cudaIpcGetMemHandle(&h, s->arena));
    memcpy(handle64, &h, 64);
    return ISB_OK;
}

int isb_shard_run_ipc_import(isb_shard_run *s, int rank, const void *handle64) {
    if (!s) return ISB_ERR_ARG;
    isb_ctx *ctx = s->model->ctx;
    ISB_LOCK(ctx);
    if (!handle64 || rank < 0 || rank >= s->G) return fail(ctx, ISB_ERR_ARG, "isb_shard_run_ipc_import: bad argument");
    if (rank == s->g) return ISB_OK;
    ISB_CUDA(ctx, cudaSetDevice(ctx->device));
    if (s->peer_open[rank]) {
        cudaIpcCloseMemHandle(s->peer_arena[rank]);
        s->peer_open[rank] = false;
    }
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    void *p = nullptr;
    ISB_CUDA(ctx, cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    s->peer_arena[rank] = (unsigned char *)p;
    s->peer_open[rank] = true;
    return ISB_OK;
}

// Signal: the epoch is written into a LOCAL staging word by a stream memory operation and copied to the flag word of
// every peer by the copy engine (stream order: after the data pushes that precede it); the wait is a stream memory
// operation on this rank's own flag words.
static int sr_signal_and_wait(isb_shard_run *s, int slot, uint64_t ep, size_t (*off_of)(const isb_shard_run *, int, int, int), int gi, int layer) {
    isb_ctx *ctx = s->model->ctx;
    if (isb::stream_write64(s->xstream, s->stage + slot, ep) != CUDA_SUCCESS)
        return fail(ctx, ISB_ERR_CUDA, "cuStreamWriteValue64 failed");
    for (int q = 0; q < s->G; ++q)
        if (q != s->g)
            ISB_CUDA(ctx, cudaMemcpyAsync(s->peer_arena[q] + off_of(s, s->g, gi, layer), s->stage + slot, sizeof(uint64_t),
                                          cudaMemcpyDeviceToDevice, s->xstream));
    for (int q = 0; q < s->G; ++q)
        if (q != s->g && isb::stream_wait_geq64(s->xstream, s->arena + off_of(s, q, gi, layer), ep) != CUDA_SUCCESS)
            return fail(ctx, ISB_ERR_CUDA, "cuStreamWaitValue64 failed (rank %d)", q);
    return ISB_OK;
}
static size_t sr_bar_off3(const isb_shard_run *s, int q, int, int) { return sr_bar_off(s, q); }

// every rank signals every peer and waits for all of them
static int sr_barrier(isb_shard_run *s) {
    isb_ctx *ctx = s->model->ctx;
    if (s->exchange != ISB_EXCH_COPY || s->G == 1) return ISB_OK;
    for (int q = 0; q < s->G; ++q)
        if (!s->peer_arena[q]) return fail(ctx, ISB_ERR_STATE, "isb_shard_run: the arena of rank %d was not imported (isb_shard_run_ipc_import)", q);
    return sr_signal_and_wait(s, SR_MAX_GROUPS * 2, ++s->bar_epoch, sr_bar_off3, 0, 0);
}

int isb_shard_run_barrier(isb_shard_run *s) {
    if (!s) return ISB_ERR_ARG;
    isb_ctx *ctx = s->model->ctx;
    ISB_LOCK(ctx);
    ISB_CUDA(ctx, cudaSetDevice(ctx->device));
    ISB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    int rc = sr_barrier(s);
    if (rc) return rc;
    ISB_CUDA(ctx, cudaStreamSynchronize(s->xstream));
    return ISB_OK;
}

int isb_shard_run_set_spins(isb_shard_run *s, const int8_t *S, int64_t ld) {
    if (!s) return ISB_ERR_ARG;
    isb_ctx *ctx = s->model->ctx;
    ISB_LOCK(ctx);
    if (!S) return fail(ctx, ISB_ERR_ARG, "isb_shard_run_set_spins: S is NULL");
    if (ld < s->n) return fail(ctx, ISB_ERR_SIZE, "isb_shard_run_set_spins: leading dimension %lld < n = %d", (long long)ld, s->n);
    for (int r = 0; r < s->R; ++r) {
        const int8_t *row = S + (int64_t)r * ld;
        unsigned bad = 0;  // branch-free so that the host compiler vectorises the scan
        for (int i = 0; i < s->n; ++i) bad |= (unsigned)((row[i] != 1) & (row[i] != -1));
        if (bad) return fail(ctx, ISB_ERR_ARG, "isb_shard_run_set_spins: replica %d holds a spin that is not +1 / -1", r);
    }
    ISB_CUDA(ctx, cudaSetDevice(ctx->device));
    ISB_CUDA(ctx, cudaStreamSynchronize(s->xstream));
    int8_t *dS = s->hostfmt;
    cudaError_t ce = cudaMemcpy2DAsync(dS, (size_t)s->n, S, (size_t)ld, (size_t)s->n, (size_t)s->R, cudaMemcpyHostToDevice, ctx->stream);
    for (int gi = 0; gi < s->ngroups && ce == cudaSuccess; ++gi) {
        SrGroup &gr = s->grp[gi];
        for (int l = 0; l < 2 && ce == cudaSuccess; ++l) {   // the embedding starts from sigma = tau = s (demo.jl:82-90)
            isb::shard_scatter_kernel<<<ctx->num_sms * 4, 256, 0, ctx->stream>>>(dS, s->n, gr.r0, gr.R, s->G, s->nb, s->esz, gr.full[l]);
            ce = cudaMemcpyAsync(gr.blk[l], (unsigned char *)gr.full[l] + (size_t)s->g * gr.R * s->nb * s->esz,
                                 (size_t)gr.R * s->nb * s->esz, cudaMemcpyDeviceToDevice, ctx->stream);
            gr.pending[l] = false;
        }
    }
    if (ce == cudaSuccess) ce = cudaGetLastError();
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(ctx->stream);
    if (ce != cudaSuccess) return fail(ctx, ISB_ERR_CUDA, "isb_shard_run_set_spins: %s", cudaGetErrorString(ce));
    // no peer may push into this rank's matrices before they hold the initial configuration
    int rc = sr_barrier(s);
    if (rc) return rc;
    ISB_CUDA(ctx, cudaStreamSynchronize(s->xstream));
    return ISB_OK;
}

int isb_shard_run_get_spins(isb_shard_run *s, int layer, int8_t *S, int64_t ld) {
    if (!s) return ISB_ERR_ARG;
    isb_ctx *ctx = s->model->ctx;
    ISB_LOCK(ctx);
    if (!S || (layer != 0 && layer != 1)) return fail(ctx, ISB_ERR_ARG, "isb_shard_run_get_spins: bad argument");
    if (ld < s->n) return fail(ctx, ISB_ERR_SIZE, "isb_shard_run_get_spins: leading dimension %lld < n = %d", (long long)ld, s->n);
    ISB_CUDA(ctx, cudaSetDevice(ctx->device));
    ISB_CUDA(ctx, cudaStreamSynchronize(s->xstream));
    int8_t *dS = s->hostfmt;
    for (int gi = 0; gi < s->ngroups; ++gi) {
        SrGroup &gr = s->grp[gi];
        isb::shard_collect_kernel<<<ctx->num_sms * 4, 256, 0, ctx->stream>>>(gr.full[layer], gr.r0, gr.R, s->G, s->nb, s->esz, dS, s->n);
    }
    cudaError_t ce = cudaGetLastError();
    if (ce == cudaSuccess)
        ce = cudaMemcpy2DAsync(S, (size_t)ld, dS, (size_t)s->n, (size_t)s->n, (size_t)s->R, cudaMemcpyDeviceToHost, ctx->stream);
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(ctx->stream);
    if (ce != cudaSuccess) return fail(ctx, ISB_ERR_CUDA, "isb_shard_run_get_spins: %s", cudaGetErrorString(ce));
    return ISB_OK;
}

int isb_shard_run_steps(isb_shard_run *s, int rule, int64_t nsteps, const double *Tsched, int64_t nT, uint64_t seed,
                        uint64_t step_offset) {
    if (!s) return ISB_ERR_ARG;
    isb_model *m = s->model;
    isb_ctx *ctx = m->ctx;
    ISB_LOCK(ctx);
    const char *who = "isb_shard_run_steps";
    if (rule != ISB_BIP_SCA && rule != ISB_BIP_MA) return fail(ctx, ISB_ERR_ARG, "%s: unknown rule %d", who, rule);
    if (nsteps < 0) return fail(ctx, ISB_ERR_ARG, "%s: nsteps is negative", who);
    if (!Tsched || nT <= 0) return fail(ctx, ISB_ERR_ARG, "%s: a temperature schedule is required", who);
    for (int64_t k = 0; k < nT; ++k)
        if (!std::isfinite(Tsched[k])) return fail(ctx, ISB_ERR_NONFINITE, "%s: non-finite temperature", who);
    isb::NcclApi *api = nullptr;
    if (s->exchange == ISB_EXCH_NCCL && s->G > 1) {
        api = isb::nccl_api();
        if (!api || !s->comm) return fail(ctx, ISB_ERR_STATE, "%s: ISB_EXCH_NCCL needs a communicator (isb_shard_run_init_nccl / _set_nccl_comm)", who);
    }
    if (s->exchange == ISB_EXCH_COPY && s->G > 1)
        for (int q = 0; q < s->G; ++q)
            if (!s->peer_arena[q]) return fail(ctx, ISB_ERR_STATE, "%s: the arena of rank %d was not imported (isb_shard_run_ipc_import)", who, q);
    ISB_CUDA(ctx, cudaSetDevice(ctx->device));
    s->launches = 0;
    ISB_CUDA(ctx, cudaEventRecord(s->ev0, ctx->stream));
    for (int64_t k = 0; k < nsteps; ++k) {
        const double T = Tsched[std::min<int64_t>(k, nT - 1)];
        for (int layer = 1; layer >= 0; --layer) {        // hidden from visible, then visible from hidden
            const int src = 1 - layer;
            for (int gi = 0; gi < s->ngroups; ++gi) {
                SrGroup &gr = s->grp[gi];
                if (gr.pending[src]) {                    // the gathered input of this half-step
                    ISB_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, gr.ready[src], 0));
                    gr.pending[src] = false;
                }
                void *own = s->G == 1 ? gr.full[layer] : gr.blk[layer];   // a single block samples in place
                ISB_TRY(isb::shard_halfstep_device(m, gr.R, gr.r0, layer, rule, gr.full[src], own, seed,
                                                   step_offset + (uint64_t)k, T));
                s->launches += 1;
                if (s->G == 1) continue;
                ISB_CUDA(ctx, cudaEventRecord(gr.sampled, ctx->stream));
                ISB_CUDA(ctx, cudaStreamWaitEvent(s->xstream, gr.sampled, 0));
                const size_t bytes = (size_t)gr.R * s->nb * s->esz;
                if (s->exchange == ISB_EXCH_NCCL) {
                    const ncclResult_t r = api->AllGather(gr.blk[layer], gr.full[layer], bytes, ncclInt8, s->comm, s->xstream);
                    if (r != ncclSuccess) return fail(ctx, ISB_ERR_NCCL, "ncclAllGather: %s", api->GetErrorString(r));
                } else {
                    const uint64_t ep = ++s->epoch[gi][layer];
                    for (int qq = 0; qq < s->G; ++qq) {   // start with the next rank: the pushes spread over the links
                        const int q = (s->g + qq) % s->G;
                        ISB_CUDA(ctx, cudaMemcpyAsync(s->peer_arena[q] + s->off_full[gi][layer] + (size_t)s->g * bytes, gr.blk[layer],
                                                      bytes, cudaMemcpyDeviceToDevice, s->xstream));
                    }
                    ISB_TRY(sr_signal_and_wait(s, gi * 2 + layer, ep, sr_flag_off, gi, layer));
                }
                ISB_CUDA(ctx, cudaEventRecord(gr.ready[layer], s->xstream));
                gr.pending[layer] = true;
            }
        }
    }
    for (int gi = 0; gi < s->ngroups; ++gi)
        for (int l = 0; l < 2; ++l)
            if (s->grp[gi].pending[l]) {
                ISB_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, s->grp[gi].ready[l], 0));
                s->grp[gi].pending[l] = false;
            }
    ISB_CUDA(ctx, cudaEventRecord(s->ev1, ctx->stream));
    cudaError_t ce = cudaStreamSynchronize(ctx->stream);
    if (ce != cudaSuccess) return fail(ctx, ISB_ERR_CUDA, "%s: kernel failed: %s", who, cudaGetErrorString(ce));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, s->ev0, s->ev1);
    s->last_ms = ms;
    return ISB_OK;
}

int isb_shard_run_last_stats(const isb_shard_run *s, double *device_ms, int64_t *launches, int *n_groups) {
    if (!s) return ISB_ERR_ARG;
    if (device_ms) *device_ms = s->last_ms;
    if (launches) *launches = s->launches;
    if (n_groups) *n_groups = s->ngroups;
    return ISB_OK;
}

}  // extern "C"
