// comm.cu — multi-GPU exchange: env-index data parallelism needs exactly one sum all-reduce of
// the flat gradient (np fp32, ~36 KB) per optimiser step plus two doubles for the global
// advantage normalisation (SURVEY §8e).  One process per GPU; the communicator is NCCL over
// NVLink 5 / NVSwitch, resolved at run time with dlopen("libnccl.so.2") so the library has no
// link-time dependency and shares the NCCL already loaded by the host process (e.g. torch's).
#include <dlfcn.h>

#include "internal.h"

namespace {
typedef struct ncclComm* ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
typedef int ncclResult_t;
enum { ncclSum = 0 };
enum { ncclFloat32 = 7, ncclFloat64 = 8 };
typedef ncclResult_t (*fn_GetUniqueId)(ncclUniqueId*);
typedef ncclResult_t (*fn_CommInitRank)(ncclComm_t*, int, ncclUniqueId, int);
typedef ncclResult_t (*fn_AllReduce)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t);
typedef ncclResult_t (*fn_CommDestroy)(ncclComm_t);
typedef const char* (*fn_GetErrorString)(ncclResult_t);

struct NcclApi {
    void* lib = nullptr;
    fn_GetUniqueId GetUniqueId = nullptr;
    fn_CommInitRank CommInitRank = nullptr;
    fn_AllReduce AllReduce = nullptr;
    fn_CommDestroy CommDestroy = nullptr;
    fn_GetErrorString GetErrorString = nullptr;
};
NcclApi g_api;

int load_nccl() {
    if (g_api.lib) return B200RL_OK;
    const char* override_path = getenv("B200RL_NCCL_LIB");
    const char* names[] = {override_path, "libnccl.so.2", "libnccl.so"};
    void* h = nullptr;
    for (const char* nm : names) {
        if (!nm) continue;
        h = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
        if (h) break;
    }
    if (!h) {
        b200rl_set_error("b200rl_comm: cannot dlopen libnccl.so.2 (%s); set B200RL_NCCL_LIB", dlerror());
        return B200RL_ERR_NCCL;
    }
    g_api.GetUniqueId = (fn_GetUniqueId)dlsym(h, "ncclGetUniqueId");
    g_api.CommInitRank = (fn_CommInitRank)dlsym(h, "ncclCommInitRank");
    g_api.AllReduce = (fn_AllReduce)dlsym(h, "ncclAllReduce");
    g_api.CommDestroy = (fn_CommDestroy)dlsym(h, "ncclCommDestroy");
    g_api.GetErrorString = (fn_GetErrorString)dlsym(h, "ncclGetErrorString");
    if (!g_api.GetUniqueId || !g_api.CommInitRank || !g_api.AllReduce || !g_api.CommDestroy) {
        b200rl_set_error("b200rl_comm: libnccl is missing required symbols");
        return B200RL_ERR_NCCL;
    }
    g_api.lib = h;
    return B200RL_OK;
}
#define NCCL_TRY(expr)                                                                                   \
    do {                                                                                                 \
        ncclResult_t _r = (expr);                                                                        \
        if (_r != 0) {                                                                                   \
            b200rl_set_error("%s -> NCCL error %d (%s)", #expr, _r, g_api.GetErrorString ? g_api.GetErrorString(_r) : "?"); \
            return B200RL_ERR_NCCL;                                                                      \
        }                                                                                                \
    } while (0)
}  // namespace

struct b200rl_comm_state {
    ncclComm_t comm;          // null when the communicator was created without NCCL (peer exchange only)
    int nranks, rank;
    unsigned char* region = nullptr;        // this rank's exchange region (cudaMalloc, exported through CUDA IPC)
    void* opened[kP2PMaxRanks] = {};        // peer regions opened with cudaIpcOpenMemHandle (closed on destroy)
    P2PTable tab = {};                      // tab.nranks > 0 once attached
    unsigned int* seq_dev = nullptr;        // device {gradient exchange, small all-reduce} sequence numbers (see common.cuh)
};

namespace {
// all-reduce (sum, in rank order => bit-identical on every rank) of a small buffer through the peer inboxes
template <class T>
__global__ void __launch_bounds__(256) p2p_allreduce_small_kernel(P2PTable tab, T* __restrict__ buf, int n, unsigned int* __restrict__ seq_ptr) {
    const unsigned seq = *seq_ptr + 1u;   // every thread reads it before the closing barrier, thread 0 stores it back after
    const unsigned slot = seq & 1u;
    constexpr int W = sizeof(T) / 4;   // 32-bit words per element
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        T mine = buf[i];
        unsigned w[2] = {0u, 0u};
        memcpy(w, &mine, sizeof(T));
        for (int h = 0; h < W; ++h) p2p_push(tab, 1, slot, (size_t)i * W + h, w[h], seq);
        T acc = 0;
        for (int r = 0; r < tab.nranks; ++r) {
            T val = mine;
            if (r != tab.rank) {
                unsigned u[2] = {0u, 0u};
                for (int h = 0; h < W; ++h) u[h] = p2p_recv(tab, 1, slot, r, (size_t)i * W + h, seq);
                memcpy(&val, u, sizeof(T));
            }
            acc += val;
        }
        buf[i] = acc;
    }
    __syncthreads();
    if (threadIdx.x == 0) *seq_ptr = seq;
}
}  // namespace

void b200rl_comm_destroy_internal(b200rl_ctx* ctx) {
    if (ctx->comm) {
        for (void* q : ctx->comm->opened) if (q) cudaIpcCloseMemHandle(q);
        if (ctx->comm->region) cudaFree(ctx->comm->region);
        if (ctx->comm->seq_dev) cudaFree(ctx->comm->seq_dev);
        if (g_api.CommDestroy && ctx->comm->comm) g_api.CommDestroy(ctx->comm->comm);
        delete ctx->comm;
        ctx->comm = nullptr;
    }
}
int b200rl_comm_world(b200rl_ctx* ctx) { return ctx->comm ? ctx->comm->nranks : 1; }
bool b200rl_comm_p2p_table(b200rl_ctx* ctx, P2PTable* out) {
    if (!ctx->comm || ctx->comm->tab.nranks <= 1) return false;
    *out = ctx->comm->tab;
    return true;
}
unsigned int* b200rl_comm_p2p_seq_dev(b200rl_ctx* ctx) { return ctx->comm ? ctx->comm->seq_dev : nullptr; }
int b200rl_comm_allreduce_internal(b200rl_ctx* ctx, void* buf, int64_t n, int is_double) {
    REQUIRE(ctx->comm, B200RL_ERR_INVALID, "no communicator");
    b200rl_comm_state* c = ctx->comm;
    if (c->tab.nranks > 1 && n * (is_double ? 2 : 1) <= (int64_t)kP2PYCap) {   // small: one kernel over NVLink peer memory
        if (is_double) p2p_allreduce_small_kernel<double><<<1, 256, 0, ctx->stream>>>(c->tab, (double*)buf, (int)n, c->seq_dev + 1);
        else p2p_allreduce_small_kernel<float><<<1, 256, 0, ctx->stream>>>(c->tab, (float*)buf, (int)n, c->seq_dev + 1);
        LAUNCH_CHECK(ctx);
        return B200RL_OK;
    }
    REQUIRE(c->comm, B200RL_ERR_UNSUPPORTED, "buffer too large for the peer exchange and no NCCL communicator");
    NCCL_TRY(g_api.AllReduce(buf, buf, (size_t)n, is_double ? ncclFloat64 : ncclFloat32, ncclSum, ctx->comm->comm, ctx->stream));
    return B200RL_OK;
}

extern "C" {
/* rank 0 creates the 128-byte NCCL unique id and ships it to the other ranks out of band */
int b200rl_comm_unique_id(void* id128_out) {
    REQUIRE(id128_out, B200RL_ERR_INVALID, "null out");
    TRY(load_nccl());
    ncclUniqueId id;
    NCCL_TRY(g_api.GetUniqueId(&id));
    memcpy(id128_out, &id, sizeof id);
    return B200RL_OK;
}
/* one process per GPU: attach ctx to rank `rank` of an `nranks` communicator */
int b200rl_comm_init(b200rl_ctx* ctx, int nranks, int rank, const void* id128) {
    TRY(ctx_bind(ctx));
    REQUIRE(nranks >= 1 && rank >= 0 && rank < nranks, B200RL_ERR_INVALID, "bad argument");
    REQUIRE(!ctx->comm, B200RL_ERR_INVALID, "communicator already initialised");
    ncclComm_t c = nullptr;
    if (id128) {   // NULL id: no NCCL, the peer exchange (b200rl_comm_p2p_*) must be attached before the first collective
        TRY(load_nccl());
        ncclUniqueId id;
        memcpy(&id, id128, sizeof id);
        NCCL_TRY(g_api.CommInitRank(&c, nranks, id, rank));
    }
    ctx->comm = new b200rl_comm_state();
    ctx->comm->comm = c; ctx->comm->nranks = nranks; ctx->comm->rank = rank;
    return B200RL_OK;
}
/* allocate this rank's exchange region; handle64_out (may be NULL) receives its CUDA IPC handle for the other processes,
 * region_out (may be NULL) the device pointer for ranks living in the same process */
int b200rl_comm_p2p_export(b200rl_ctx* ctx, void* handle64_out, void** region_out) {
    TRY(ctx_bind(ctx));
    REQUIRE(ctx->comm, B200RL_ERR_INVALID, "b200rl_comm_init first");
    b200rl_comm_state* c = ctx->comm;
    if (!c->region) {
        CUDA_TRY(cudaMalloc(&c->region, kP2PRegionBytes));
        CUDA_TRY(cudaMemset(c->region, 0, kP2PRegionBytes));
        CUDA_TRY(cudaMalloc(&c->seq_dev, 2 * sizeof(unsigned int)));
        CUDA_TRY(cudaMemset(c->seq_dev, 0, 2 * sizeof(unsigned int)));
        CUDA_TRY(cudaDeviceSynchronize());
    }
    if (handle64_out) {
        static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
        cudaIpcMemHandle_t h;
        CUDA_TRY(cudaIpcGetMemHandle(&h, c->region));
        memcpy(handle64_out, &h, sizeof h);
    }
    if (region_out) *region_out = c->region;
    return B200RL_OK;
}
/* map another process's region (its 64-byte IPC handle) into this process */
int b200rl_comm_p2p_open(b200rl_ctx* ctx, const void* handle64, void** region_out) {
    TRY(ctx_bind(ctx));
    REQUIRE(ctx->comm && handle64 && region_out, B200RL_ERR_INVALID, "bad argument");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, sizeof h);
    void* q = nullptr;
    CUDA_TRY(cudaIpcOpenMemHandle(&q, h, cudaIpcMemLazyEnablePeerAccess));
    for (void*& slot : ctx->comm->opened) if (!slot) { slot = q; break; }
    *region_out = q;
    return B200RL_OK;
}
/* regions[r] = device pointer of rank r's region as seen by THIS process (entry `rank` may be NULL: own region).
 * From here on gradient and small all-reduces go through peer memory in one fused kernel each. */
int b200rl_comm_p2p_attach(b200rl_ctx* ctx, void* const* regions) {
    TRY(ctx_bind(ctx));
    REQUIRE(ctx->comm && regions, B200RL_ERR_INVALID, "bad argument");
    b200rl_comm_state* c = ctx->comm;
    REQUIRE(c->region, B200RL_ERR_INVALID, "b200rl_comm_p2p_export first");
    REQUIRE(c->nranks <= kP2PMaxRanks, B200RL_ERR_UNSUPPORTED, "peer exchange supports up to 8 ranks (one NVSwitch node)");
    P2PTable t = {};
    t.nranks = c->nranks; t.rank = c->rank;
    t.exclusive = 1;
    for (int r = 0; r < c->nranks; ++r) {
        t.base[r] = r == c->rank ? c->region : (unsigned char*)regions[r];
        REQUIRE(t.base[r], B200RL_ERR_INVALID, "null peer region");
        if (r != c->rank) {   // same-process peers on another device: enable direct access (IPC mappings already are)
            cudaPointerAttributes at;
            if (cudaPointerGetAttributes(&at, t.base[r]) == cudaSuccess) {
                if (at.device != ctx->device) {
                    cudaError_t e = cudaDeviceEnablePeerAccess(at.device, 0);
                    if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); }
                    else cudaGetLastError();
                } else {
                    t.exclusive = 0;   // a peer rank drives this very device
                }
            } else {
                cudaGetLastError();
                t.exclusive = 0;
            }
        }
    }
    c->tab = t;
    return B200RL_OK;
}
int b200rl_ctx_pci_bus_id(b200rl_ctx* ctx, char* out, int len) {
    TRY(ctx_bind(ctx));
    REQUIRE(out && len >= 16, B200RL_ERR_INVALID, "bad argument");
    CUDA_TRY(cudaDeviceGetPCIBusId(out, len, ctx->device));
    return B200RL_OK;
}
int b200rl_comm_p2p_set_exclusive(b200rl_ctx* ctx, int exclusive) {
    REQUIRE(ctx && ctx->comm && ctx->comm->tab.nranks > 1, B200RL_ERR_INVALID, "attach the peer exchange first");
    ctx->comm->tab.exclusive = exclusive ? 1 : 0;
    return B200RL_OK;
}
/* in-place sum all-reduce of a DEVICE fp32 buffer on the ctx stream */
int b200rl_comm_allreduce_f32(b200rl_ctx* ctx, float* dev_buf, int64_t n) {
    TRY(ctx_bind(ctx));
    REQUIRE(dev_buf && n > 0, B200RL_ERR_INVALID, "bad argument");
    return b200rl_comm_allreduce_internal(ctx, dev_buf, n, 0);
}
}
