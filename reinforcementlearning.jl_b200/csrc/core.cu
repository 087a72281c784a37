// core.cu — context, error convention, memory helpers of libb200rl.so.
#include <cstdarg>
#include <cstdlib>

#include "internal.h"

static thread_local char g_err[1024] = "no error";

void b200rl_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
}

int ctx_scratch(b200rl_ctx* ctx, size_t bytes, void** out) {
    if (bytes > ctx->scratch_bytes) {
        // The old buffer may still be read by queued work, and cudaFree would synchronise the whole device (a deadlock when
        // another rank of the same process is spinning on this rank inside the peer exchange): retire it, free at destroy.
        if (ctx->scratch) ctx->retired.push_back(ctx->scratch);
        ctx->scratch = nullptr;
        ctx->scratch_bytes = 0;
        size_t want = bytes + bytes / 4 + 4096;
        CUDA_TRY(cudaMalloc(&ctx->scratch, want));
        ctx->scratch_bytes = want;
    }
    *out = ctx->scratch;
    return B200RL_OK;
}

__global__ void flush_kernel(float4* p, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t stride = (size_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) p[i] = make_float4(1.f, 2.f, 3.f, 4.f);
}

extern "C" {

const char* b200rl_last_error(void) { return g_err; }
int b200rl_abi_version(void) { return B200RL_ABI_VERSION; }

int b200rl_init(int device, b200rl_ctx** out) {
    REQUIRE(out, B200RL_ERR_INVALID, "null out");
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        b200rl_set_error("b200rl_init: no CUDA device visible (%s); this library has no CPU fallback",
                         e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
        return B200RL_ERR_CUDA;
    }
    REQUIRE(device >= 0 && device < count, B200RL_ERR_INVALID, "device index out of range");
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        b200rl_set_error("b200rl_init: device %d is sm_%d%d; libb200rl.so contains sm_100a code only", device, prop.major, prop.minor);
        return B200RL_ERR_UNSUPPORTED;
    }
    CUDA_TRY(cudaSetDevice(device));
    {   // L2 fetch granularity 32 B: the minibatch gathers of the update read one 32-byte record per sample at random; with the
        // default (128 B) granularity every such read drags 3 neighbouring sectors out of HBM (ncu: 46.0 MB per K7 launch vs
        // 16.9 MB at 32 B = 1.01x the algorithmic bytes; streaming kernels request whole lines either way).  A hint, per context;
        // B200RL_L2_FETCH=64|128 restores a larger one, 0 leaves the driver default.
        size_t gran = 32;
        if (const char* g = getenv("B200RL_L2_FETCH")) gran = (size_t)atoi(g);
        if (gran) { cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, gran); cudaGetLastError(); }
    }
    b200rl_ctx* ctx = new b200rl_ctx();
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    ctx->l2_bytes = (size_t)prop.l2CacheSize;
    CUDA_TRY(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    CUDA_TRY(cudaEventCreate(&ctx->ev0));
    CUDA_TRY(cudaEventCreate(&ctx->ev1));
    *out = ctx;
    return B200RL_OK;
}

void b200rl_destroy(b200rl_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    b200rl_comm_destroy_internal(ctx);
    if (ctx->scratch) cudaFree(ctx->scratch);
    for (void* q : ctx->retired) cudaFree(q);
    if (ctx->flush_buf) cudaFree(ctx->flush_buf);
    cudaEventDestroy(ctx->ev0);
    cudaEventDestroy(ctx->ev1);
    for (cudaEvent_t e : ctx->slots) if (e) cudaEventDestroy(e);
    cudaStreamDestroy(ctx->stream);
    delete ctx;
}

int b200rl_sync(b200rl_ctx* ctx) {
    TRY(ctx_bind(ctx));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return B200RL_OK;
}
int b200rl_stream(b200rl_ctx* ctx, void** stream_out) {
    REQUIRE(ctx && stream_out, B200RL_ERR_INVALID, "null argument");
    *stream_out = (void*)ctx->stream;
    return B200RL_OK;
}
int b200rl_launch_count(b200rl_ctx* ctx, uint64_t* out) {
    REQUIRE(ctx && out, B200RL_ERR_INVALID, "null argument");
    *out = ctx->launches;
    return B200RL_OK;
}
int b200rl_timer_start(b200rl_ctx* ctx) {
    TRY(ctx_bind(ctx));
    CUDA_TRY(cudaEventRecord(ctx->ev0, ctx->stream));
    return B200RL_OK;
}
int b200rl_timer_stop_ms(b200rl_ctx* ctx, float* ms_out) {
    TRY(ctx_bind(ctx));
    REQUIRE(ms_out, B200RL_ERR_INVALID, "null out");
    CUDA_TRY(cudaEventRecord(ctx->ev1, ctx->stream));
    CUDA_TRY(cudaEventSynchronize(ctx->ev1));
    CUDA_TRY(cudaEventElapsedTime(ms_out, ctx->ev0, ctx->ev1));
    return B200RL_OK;
}
/* event slots: record any number of points on the ctx stream without synchronising, read the intervals afterwards */
int b200rl_timer_record(b200rl_ctx* ctx, int slot) {
    TRY(ctx_bind(ctx));
    REQUIRE(slot >= 0 && slot < b200rl_ctx::kTimerSlots, B200RL_ERR_INVALID, "timer slot out of range");
    if (!ctx->slots[slot]) CUDA_TRY(cudaEventCreate(&ctx->slots[slot]));
    CUDA_TRY(cudaEventRecord(ctx->slots[slot], ctx->stream));
    return B200RL_OK;
}
int b200rl_timer_elapsed_ms(b200rl_ctx* ctx, int slot_from, int slot_to, float* ms_out) {
    TRY(ctx_bind(ctx));
    REQUIRE(ms_out && slot_from >= 0 && slot_from < b200rl_ctx::kTimerSlots && slot_to >= 0 && slot_to < b200rl_ctx::kTimerSlots,
            B200RL_ERR_INVALID, "bad argument");
    REQUIRE(ctx->slots[slot_from] && ctx->slots[slot_to], B200RL_ERR_INVALID, "timer slot never recorded");
    CUDA_TRY(cudaEventSynchronize(ctx->slots[slot_to]));
    CUDA_TRY(cudaEventElapsedTime(ms_out, ctx->slots[slot_from], ctx->slots[slot_to]));
    return B200RL_OK;
}
/* measurement aid: base_slot >= 0 makes b200rl_onpolicy_update (eager path) record its phases into the timer slots
 * base_slot + {0: entry, 1: after GAE / normalisation / packing, 2 + 2i: after loss+backward i, 3 + 2i: after optimiser step i};
 * -1 switches it off */
int b200rl_debug_phase_slots(b200rl_ctx* ctx, int base_slot) {
    REQUIRE(ctx && base_slot >= -1 && base_slot < b200rl_ctx::kTimerSlots - 8, B200RL_ERR_INVALID, "bad argument");
    ctx->phase_base = base_slot;
    return B200RL_OK;
}
int b200rl_malloc(b200rl_ctx* ctx, size_t bytes, void** dptr_out) {
    TRY(ctx_bind(ctx));
    REQUIRE(dptr_out, B200RL_ERR_INVALID, "null out");
    CUDA_TRY(cudaMalloc(dptr_out, bytes ? bytes : 1));
    return B200RL_OK;
}
int b200rl_free(b200rl_ctx* ctx, void* dptr) {
    TRY(ctx_bind(ctx));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    CUDA_TRY(cudaFree(dptr));
    return B200RL_OK;
}
int b200rl_host_alloc(b200rl_ctx* ctx, size_t bytes, void** hptr_out) {
    TRY(ctx_bind(ctx));
    REQUIRE(hptr_out, B200RL_ERR_INVALID, "null out");
    CUDA_TRY(cudaHostAlloc(hptr_out, bytes ? bytes : 1, cudaHostAllocDefault));
    return B200RL_OK;
}
int b200rl_host_free(b200rl_ctx* ctx, void* hptr) {
    TRY(ctx_bind(ctx));
    CUDA_TRY(cudaFreeHost(hptr));
    return B200RL_OK;
}
int b200rl_memcpy_h2d(b200rl_ctx* ctx, void* dst, const void* src, size_t bytes, int async) {
    TRY(ctx_bind(ctx));
    CUDA_TRY(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    if (!async) CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return B200RL_OK;
}
int b200rl_memcpy_d2h(b200rl_ctx* ctx, void* dst, const void* src, size_t bytes, int async) {
    TRY(ctx_bind(ctx));
    CUDA_TRY(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    if (!async) CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return B200RL_OK;
}
int b200rl_memset(b200rl_ctx* ctx, void* dst, int value, size_t bytes) {
    TRY(ctx_bind(ctx));
    CUDA_TRY(cudaMemsetAsync(dst, value, bytes, ctx->stream));
    return B200RL_OK;
}
int b200rl_flush_l2(b200rl_ctx* ctx) {
    TRY(ctx_bind(ctx));
    if (!ctx->flush_buf) {
        ctx->flush_bytes = ctx->l2_bytes * 2 > ((size_t)256 << 20) ? ctx->l2_bytes * 2 : ((size_t)256 << 20);
        CUDA_TRY(cudaMalloc(&ctx->flush_buf, ctx->flush_bytes));
    }
    flush_kernel<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>((float4*)ctx->flush_buf, ctx->flush_bytes / 16);
    CUDA_TRY(cudaGetLastError());  // not counted in ctx->launches: bench hygiene, not hot path
    return B200RL_OK;
}

}  // extern "C"
