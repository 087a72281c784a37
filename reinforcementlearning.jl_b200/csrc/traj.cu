// traj.cu — K3/K4: device-resident trajectory ring (CircularArraySARTSTraces), push!, and
// uniform / prioritised minibatch sampling + gather.
//
// Upstream = ReinforcementLearningTrajectories 0.4 (not vendored; SURVEY Appendix B); anchored
// on the reference's call sites: push order agent_base.jl:45-59 / agent_srt_cache.jl:30-50,
// trace layout docs/src/How_to_implement_a_new_algorithm.md:84-112, length semantics
// RLCore/test/policies/agent.jl:27-34, iteration tuple test/policies/q_based_policy.jl:40-58.
//
// Layout in HBM: cap+1 slots per lane, slot-major so that lanes at the same ring position are contiguous:
//   state (ns, lanes, cap+1) f32 | action (lanes, cap+1) i32 | reward (lanes, cap+1) f32 |
//   flag (lanes, cap+1) u8 (bit0 terminal, bit1 sampleable) | sum tree 2L f32 (leaf = slot*lanes + lane).
// Entry p of a lane is the transition state[p] -> state[p+1] (MultiplexTraces without a second copy).
// EpisodesBuffer semantics PER LANE (RLTrajectories 0.4; pinned by RLCore/test/core/base.jl:20: length == steps + episodes - 1):
// every lane has its own ring position (head) and fill level (count).  The first state of an episode is a frame of its own
// (push_episode_start, the PreEpisodeStage push of agent_base.jl:45-47), so the entry that straddles two episodes exists, counts
// towards length(container) and is never sampleable.  With the env's in-kernel auto-reset the terminal step's next observation
// already is the new episode's first state: the push stores it twice (as the masked :next_state of the terminal entry and as
// the episode-start frame), which reproduces the reference's entry count and sampleable set exactly.
// A push is one thread per lane (neighbouring lanes write neighbouring addresses unless their episode counts differ);
// a sample is one thread per batch slot: Xoshiro draw -> (rejection | sum-tree descent) -> 2 x state gather + scalars.
#include "internal.h"

namespace {

struct Xo4 { unsigned long long s[4]; };
__device__ __forceinline__ Xo4 load_xo(const unsigned long long* rng, int64_t i) {
    const ulonglong2* p = reinterpret_cast<const ulonglong2*>(rng + 4 * i);
    ulonglong2 a = p[0], b = p[1];
    Xo4 g; g.s[0] = a.x; g.s[1] = a.y; g.s[2] = b.x; g.s[3] = b.y;
    return g;
}
__device__ __forceinline__ void store_xo(unsigned long long* rng, int64_t i, const Xo4& g) {
    ulonglong2* p = reinterpret_cast<ulonglong2*>(rng + 4 * i);
    p[0] = make_ulonglong2(g.s[0], g.s[1]);
    p[1] = make_ulonglong2(g.s[2], g.s[3]);
}
__device__ __forceinline__ unsigned long long xo_next(Xo4& g) {
    unsigned long long tmp = g.s[0] + g.s[3];
    unsigned long long res = ((tmp << 23) | (tmp >> 41)) + g.s[0];
    unsigned long long t = g.s[1] << 17;
    g.s[2] ^= g.s[0]; g.s[3] ^= g.s[1]; g.s[1] ^= g.s[2]; g.s[0] ^= g.s[3]; g.s[2] ^= t;
    g.s[3] = (g.s[3] << 45) | (g.s[3] >> 19);
    return res;
}
// rand(rng, Base.OneTo(n)) - 1  (Lemire nearly-divisionless, Julia SamplerRangeNDL)
__device__ __forceinline__ unsigned long long rand_below(Xo4& g, unsigned long long n) {
    unsigned long long x = xo_next(g);
    unsigned long long hi = __umul64hi(x, n), lo = x * n;
    if (lo < n) {
        unsigned long long t = (0ull - n) % n;
        while (lo < t) { x = xo_next(g); hi = __umul64hi(x, n); lo = x * n; }
    }
    return hi;
}

struct Ring {
    int ns;
    int64_t lanes, cap;
    float* state; int32_t* action; float* reward; uint8_t* flag;
    int32_t* head;       // (lanes) next slot to write
    int32_t* count;      // (lanes) state frames stored, <= cap + 1
    uint8_t* pending;    // (lanes) the last stored transition was terminal and its episode-start frame has not been pushed yet
    long long* n_valid;  // (1) sampleable entries over all lanes
    float* tree; int64_t L;
    __host__ __device__ int64_t frames() const { return cap + 1; }
};
constexpr uint8_t kTerminal = 1, kSampleable = 2;

// ---- push kernels: one thread per lane; `keys`/`vals` (3 per lane) receive the sum-tree leaves to rewrite (key -1 = none) --------
__device__ __forceinline__ void write_state(const Ring& r, int64_t slot, int64_t e, const float* __restrict__ obs) {
    float* dst = r.state + (int64_t)r.ns * (slot * r.lanes + e);
    const float* src = obs + (int64_t)r.ns * e;
    for (int c = 0; c < r.ns; ++c) dst[c] = src[c];
}
// the state frame at `slot` is about to be overwritten: the entry that started there is gone
__device__ __forceinline__ int destroy_entry(const Ring& r, int64_t slot, int64_t e) {
    const int64_t k = slot * r.lanes + e;
    const int was = (r.flag[k] & kSampleable) ? 1 : 0;
    r.flag[k] = 0;
    return was;
}
// push!(trajectory, (state = s0,)): mode 0 every lane, 1 only lanes whose last transition was terminal (soft reset)
__global__ void push_episode_start_kernel(Ring r, const float* __restrict__ obs, int mode, float default_priority, int64_t* __restrict__ keys,
                                          float* __restrict__ vals) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= r.lanes) return;
    if (keys) { keys[3 * e] = -1; keys[3 * e + 1] = -1; keys[3 * e + 2] = -1; }
    if (mode == 1 && !r.pending[e]) return;
    const int64_t F = r.frames();
    const int64_t h = r.head[e];
    const int lost = destroy_entry(r, h, e);
    write_state(r, h, e, obs);
    if (keys) { keys[3 * e] = h * r.lanes + e; vals[3 * e] = 0.f; }
    r.head[e] = (int32_t)((h + 1) % F);
    r.count[e] = (int32_t)min((int64_t)r.count[e] + 1, F);
    r.pending[e] = 0;
    if (lost) atomicAdd((unsigned long long*)r.n_valid, (unsigned long long)(-1ll));
}
// push!(trajectory, (state = s', action, reward, terminal)).  term[e]: bit0 terminal, bit1 "the env has already auto-reset: next_obs
// is the first state of the next episode" (the env's FLAGS byte) -> the episode-start frame is written in the same launch.
__global__ void push_sart_kernel(Ring r, const int32_t* __restrict__ a, const float* __restrict__ rew, const uint8_t* __restrict__ term,
                                 const float* __restrict__ next_obs, float default_priority, int64_t* __restrict__ keys, float* __restrict__ vals) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= r.lanes) return;
    const int64_t F = r.frames();
    const int64_t h = r.head[e];
    const int64_t p = (h + F - 1) % F;                 // slot of the state the action was taken in
    const uint8_t t = term[e];
    r.action[p * r.lanes + e] = a[e];
    r.reward[p * r.lanes + e] = rew[e];
    r.flag[p * r.lanes + e] = (uint8_t)((t & kTerminal) | kSampleable);
    long long dv = 1;
    dv -= destroy_entry(r, h, e);
    write_state(r, h, e, next_obs);
    int64_t nh = (h + 1) % F;
    int cnt = (int)min((int64_t)r.count[e] + 1, F);
    if (keys) {
        keys[3 * e] = p * r.lanes + e; vals[3 * e] = default_priority;
        keys[3 * e + 1] = h * r.lanes + e; vals[3 * e + 1] = 0.f;
        keys[3 * e + 2] = -1;
    }
    uint8_t pend = 0;
    if (t & kTerminal) {
        if (t & 2) {                                   // auto-reset: next_obs doubles as the episode-start frame
            dv -= destroy_entry(r, nh, e);
            write_state(r, nh, e, next_obs);
            if (keys) { keys[3 * e + 2] = nh * r.lanes + e; vals[3 * e + 2] = 0.f; }
            nh = (nh + 1) % F;
            cnt = (int)min((int64_t)cnt + 1, F);
        } else {
            pend = 1;                                  // the caller pushes the episode start once the env has been reset
        }
    }
    r.head[e] = (int32_t)nh;
    r.count[e] = cnt;
    r.pending[e] = pend;
    if (dv != 0) atomicAdd((unsigned long long*)r.n_valid, (unsigned long long)dv);
}

// Single CTA: tree[L + key[k]] = prio[k] for every key >= 0, then rebuild the touched paths level by level
// (children are re-added, never delta-updated -> deterministic, drift-free; duplicate keys must carry one value).
// The levels below node 4096 are walked per key (global memory, one dependent round trip per level); the top 12 levels
// (nodes 1..4095, shared by every path) are rebuilt wholesale in shared memory from the 4096 nodes below them — the same
// pairwise sums, so the tree is bit-identical to the level-by-level walk, at a fraction of the dependent-latency chain.
constexpr int kTopNodes = 4096;
__global__ void __launch_bounds__(1024) tree_update_keys_kernel(float* __restrict__ tree, int64_t L, const int64_t* __restrict__ key,
                                                                const float* __restrict__ prio, int64_t B) {
    __shared__ float top[2 * kTopNodes];     // top[n] = node n for n < 2 * kTopNodes (children level loaded, the rest computed)
    for (int64_t k = threadIdx.x; k < B; k += blockDim.x)
        if (key[k] >= 0) tree[L + key[k]] = prio[k];
    __syncthreads();
    int shift = 1;
    for (; (L >> shift) >= kTopNodes; ++shift) {  // nodes >= kTopNodes: one tree level per iteration, leaves' parents first
        for (int64_t k = threadIdx.x; k < B; k += blockDim.x) {
            if (key[k] < 0) continue;
            int64_t node = (L + key[k]) >> shift;
            tree[node] = tree[2 * node] + tree[2 * node + 1];
        }
        __syncthreads();
    }
    if (L >= kTopNodes) {
        // (L >> shift) == kTopNodes / 2: nodes [kTopNodes, 2 kTopNodes) are final; everything above is recomputed from them
        for (int n = threadIdx.x; n < kTopNodes; n += blockDim.x) top[kTopNodes + n] = tree[kTopNodes + n];
        __syncthreads();
        for (int width = kTopNodes / 2; width >= 1; width >>= 1) {
            for (int n = threadIdx.x; n < width; n += blockDim.x) top[width + n] = top[2 * (width + n)] + top[2 * (width + n) + 1];
            __syncthreads();
        }
        for (int n = 1 + threadIdx.x; n < kTopNodes; n += blockDim.x) tree[n] = top[n];
    } else {
        for (; (L >> shift) >= 1; ++shift) {
            for (int64_t k = threadIdx.x; k < B; k += blockDim.x) {
                if (key[k] < 0) continue;
                int64_t node = (L + key[k]) >> shift;
                tree[node] = tree[2 * node] + tree[2 * node + 1];
            }
            __syncthreads();
        }
    }
}

struct BatchOut {
    float* s; int32_t* a; float* r; uint8_t* t; float* s2; int64_t* key; float* prio; float* w;
};

// The descent of the binary sum tree is a chain of dependent reads (20 levels for 1 M leaves): the top kTopLevels levels
// (nodes 1 .. 2^kTopLevels - 1, 16 KB) are staged in shared memory by the CTA with independent loads, which leaves 8 dependent
// L2 round trips instead of 20; a node's two children are adjacent and read as one 8-byte word.  Same values, same comparisons.
constexpr int kTopLevels = 12;
template <bool PRIO>
__global__ void __launch_bounds__(128) sample_gather_kernel(Ring r, unsigned long long* __restrict__ slots, int64_t B, float beta, BatchOut o) {
    __shared__ float top[PRIO ? (1 << kTopLevels) : 1];
    if (PRIO) {
        const int64_t ntop = min((int64_t)(1 << kTopLevels), 2 * r.L);
        for (int64_t i = threadIdx.x; i < ntop; i += blockDim.x) top[i] = r.tree[i];
        __syncthreads();
    }
    int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= B) return;
    Xo4 g = load_xo(slots, k);
    const int64_t F = r.frames();
    int64_t key;
    float p = 0.f, w = 1.f;
    if (PRIO) {
        const float total = top[1];
        float v = ((float)((unsigned)(xo_next(g) >> 32) >> 8) * 0x1p-24f) * total;  // rand(rng, Float32) * total
        int64_t node = 1;
        while (node < r.L) {     // never step into an empty subtree: float rounding cannot land on a zero-priority leaf
            const int64_t l = 2 * node;
            float tl, tr;
            if (l + 1 < (1 << kTopLevels)) { tl = top[l]; tr = top[l + 1]; }
            else { const float2 c2 = *reinterpret_cast<const float2*>(r.tree + l); tl = c2.x; tr = c2.y; }
            if (tl > 0.f && (v < tl || !(tr > 0.f))) node = l;
            else { v -= tl; node = l + 1; }
        }
        key = node - r.L;
        p = r.tree[r.L + key];
        const long long n = *r.n_valid;
        w = powf((float)n * (p / total), -beta);
    } else {
        // uniform over the sampleable entries: draw (lane, logical index) and redraw while it is not one
        const unsigned long long n = (unsigned long long)(r.lanes * r.cap);
        key = -1;
        for (int tries = 0; tries < 4096; ++tries) {
            const int64_t q = (int64_t)rand_below(g, n);
            const int64_t e = q % r.lanes, j = q / r.lanes;
            const int64_t cnt = r.count[e];
            if (j >= cnt - 1) continue;
            const int64_t slot = ((int64_t)r.head[e] - cnt + j + 2 * F) % F;
            if (r.flag[slot * r.lanes + e] & kSampleable) { key = slot * r.lanes + e; break; }
        }
        if (key < 0) __trap();   // (practically) nothing sampleable
    }
    store_xo(slots, k, g);
    const int64_t slot = key / r.lanes, e = key % r.lanes;
    const int64_t nslot = (slot + 1) % F;
    const float* s = r.state + (int64_t)r.ns * (slot * r.lanes + e);
    const float* s2 = r.state + (int64_t)r.ns * (nslot * r.lanes + e);
    if (r.ns == 4) {   // one 16-byte row each way
        reinterpret_cast<float4*>(o.s)[k] = *reinterpret_cast<const float4*>(s);
        reinterpret_cast<float4*>(o.s2)[k] = *reinterpret_cast<const float4*>(s2);
    } else {
        for (int c = 0; c < r.ns; ++c) { o.s[(int64_t)r.ns * k + c] = s[c]; o.s2[(int64_t)r.ns * k + c] = s2[c]; }
    }
    o.a[k] = r.action[key];
    o.r[k] = r.reward[key];
    o.t[k] = r.flag[key] & kTerminal;
    o.key[k] = key;
    o.prio[k] = p;
    o.w[k] = w;
}
// w /= max(w) (single CTA, fixed tree)
__global__ void __launch_bounds__(1024) normalize_weights_kernel(float* __restrict__ w, int64_t B) {
    __shared__ float red[32];
    float m = 0.f;
    for (int64_t k = threadIdx.x; k < B; k += blockDim.x) m = fmaxf(m, w[k]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
    __syncthreads();
    m = 0.f;
    for (int k = 0; k < (int)(blockDim.x >> 5); ++k) m = fmaxf(m, red[k]);
    for (int64_t k = threadIdx.x; k < B; k += blockDim.x) w[k] = w[k] / m;
}
// new priorities from TD errors: (|td| + eps)^alpha   (PrioritizedDQN, SURVEY Appendix B)
__global__ void td_to_priority_kernel(const float* __restrict__ td, float* __restrict__ prio, int64_t B, float eps, float alpha) {
    int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < B) prio[k] = powf(fabsf(td[k]) + eps, alpha);
}

}  // namespace

struct b200rl_traj {
    b200rl_ctx* ctx;
    Ring r;
    bool prioritized;
    float default_priority;
    int64_t B;
    unsigned long long* slots;  // (4, B) sampler streams
    BatchOut batch;
    float* new_prio;            // (B) scratch for priority write-back
    int64_t* keys; float* vals; // (3 * lanes) sum-tree leaves rewritten by a push
    void* stage;                // staging for host-side pushes
    size_t stage_bytes;
    int64_t pushed;             // transitions frames pushed so far (host-side sanity only)
};

static int stage_in(b200rl_traj* t, const void* host, size_t bytes, size_t offset, const void** dev) {
    REQUIRE(offset + bytes <= t->stage_bytes, B200RL_ERR_INVALID, "staging overflow");
    CUDA_TRY(cudaMemcpyAsync((char*)t->stage + offset, host, bytes, cudaMemcpyHostToDevice, t->ctx->stream));
    *dev = (char*)t->stage + offset;
    return B200RL_OK;
}
static int tree_apply(b200rl_traj* t) {
    if (!t->prioritized) return B200RL_OK;
    tree_update_keys_kernel<<<1, 1024, 0, t->ctx->stream>>>(t->r.tree, t->r.L, t->keys, t->vals, 3 * t->r.lanes);
    LAUNCH_CHECK(t->ctx);
    return B200RL_OK;
}

extern "C" {

int b200rl_traj_create(b200rl_ctx* ctx, int ns, int64_t lanes, int64_t capacity, int prioritized, float default_priority,
                       const uint64_t* sampler_rng, int64_t batch_size, b200rl_traj** out) {
    TRY(ctx_bind(ctx));
    REQUIRE(out && ns >= 1 && ns <= 16 && lanes >= 1 && capacity >= 2, B200RL_ERR_INVALID, "bad shape (capacity >= 2)");
    REQUIRE(batch_size >= 0 && (batch_size == 0 || sampler_rng), B200RL_ERR_INVALID, "sampler_rng required when batch_size > 0");
    REQUIRE((capacity + 1) < (1ll << 31), B200RL_ERR_UNSUPPORTED, "capacity too large");
    b200rl_traj* t = new b200rl_traj();
    memset(t, 0, sizeof *t);
    t->ctx = ctx; t->prioritized = prioritized != 0; t->default_priority = default_priority; t->B = batch_size;
    Ring& r = t->r;
    r.ns = ns; r.lanes = lanes; r.cap = capacity;
    size_t slots = (size_t)lanes * (capacity + 1);
    CUDA_TRY(cudaMalloc(&r.state, slots * ns * sizeof(float)));
    CUDA_TRY(cudaMalloc(&r.action, slots * sizeof(int32_t)));
    CUDA_TRY(cudaMalloc(&r.reward, slots * sizeof(float)));
    CUDA_TRY(cudaMalloc(&r.flag, slots));
    CUDA_TRY(cudaMalloc(&r.head, (size_t)lanes * 4)); CUDA_TRY(cudaMalloc(&r.count, (size_t)lanes * 4)); CUDA_TRY(cudaMalloc(&r.pending, (size_t)lanes));
    CUDA_TRY(cudaMalloc(&r.n_valid, 8));
    CUDA_TRY(cudaMemsetAsync(r.state, 0, slots * ns * sizeof(float), ctx->stream));
    CUDA_TRY(cudaMemsetAsync(r.action, 0, slots * 4, ctx->stream)); CUDA_TRY(cudaMemsetAsync(r.reward, 0, slots * 4, ctx->stream));
    CUDA_TRY(cudaMemsetAsync(r.flag, 0, slots, ctx->stream));
    CUDA_TRY(cudaMemsetAsync(r.head, 0, (size_t)lanes * 4, ctx->stream)); CUDA_TRY(cudaMemsetAsync(r.count, 0, (size_t)lanes * 4, ctx->stream));
    CUDA_TRY(cudaMemsetAsync(r.pending, 0, (size_t)lanes, ctx->stream)); CUDA_TRY(cudaMemsetAsync(r.n_valid, 0, 8, ctx->stream));
    r.L = 1;
    if (t->prioritized) {
        while (r.L < (int64_t)slots) r.L <<= 1;
        CUDA_TRY(cudaMalloc(&r.tree, 2 * r.L * sizeof(float)));
        CUDA_TRY(cudaMemsetAsync(r.tree, 0, 2 * r.L * sizeof(float), ctx->stream));
        CUDA_TRY(cudaMalloc(&t->keys, (size_t)lanes * 3 * 8)); CUDA_TRY(cudaMalloc(&t->vals, (size_t)lanes * 3 * 4));
    }
    if (batch_size > 0) {
        size_t B = (size_t)batch_size;
        CUDA_TRY(cudaMalloc(&t->slots, B * 32));
        CUDA_TRY(cudaMemcpyAsync(t->slots, sampler_rng, B * 32, cudaMemcpyHostToDevice, ctx->stream));
        CUDA_TRY(cudaMalloc(&t->batch.s, B * ns * sizeof(float)));
        CUDA_TRY(cudaMalloc(&t->batch.s2, B * ns * sizeof(float)));
        CUDA_TRY(cudaMalloc(&t->batch.a, B * 4));
        CUDA_TRY(cudaMalloc(&t->batch.r, B * 4));
        CUDA_TRY(cudaMalloc(&t->batch.t, B));
        CUDA_TRY(cudaMalloc(&t->batch.key, B * 8));
        CUDA_TRY(cudaMalloc(&t->batch.prio, B * 4));
        CUDA_TRY(cudaMalloc(&t->batch.w, B * 4));
        CUDA_TRY(cudaMalloc(&t->new_prio, B * 4));
    }
    t->stage_bytes = (size_t)lanes * (ns * 4 + 4 + 4 + 1) + 64;
    CUDA_TRY(cudaMalloc(&t->stage, t->stage_bytes));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    *out = t;
    return B200RL_OK;
}

int b200rl_traj_destroy(b200rl_traj* t) {
    if (!t) return B200RL_OK;
    cudaSetDevice(t->ctx->device);
    cudaStreamSynchronize(t->ctx->stream);
    cudaFree(t->r.state); cudaFree(t->r.action); cudaFree(t->r.reward); cudaFree(t->r.flag); cudaFree(t->r.tree);
    cudaFree(t->r.head); cudaFree(t->r.count); cudaFree(t->r.pending); cudaFree(t->r.n_valid); cudaFree(t->keys); cudaFree(t->vals);
    cudaFree(t->slots); cudaFree(t->batch.s); cudaFree(t->batch.s2); cudaFree(t->batch.a); cudaFree(t->batch.r); cudaFree(t->batch.t);
    cudaFree(t->batch.key); cudaFree(t->batch.prio); cudaFree(t->batch.w); cudaFree(t->new_prio); cudaFree(t->stage);
    delete t;
    return B200RL_OK;
}

/* length(trajectory.container) per lane: entries stored (sampleable or not) = state frames - 1 (synchronises) */
int b200rl_traj_lane_lengths(b200rl_traj* t, int64_t* lengths_out) {
    REQUIRE(t && lengths_out, B200RL_ERR_INVALID, "null argument");
    TRY(ctx_bind(t->ctx));
    std::vector<int32_t> c((size_t)t->r.lanes);
    CUDA_TRY(cudaMemcpyAsync(c.data(), t->r.count, c.size() * 4, cudaMemcpyDeviceToHost, t->ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(t->ctx->stream));
    for (int64_t e = 0; e < t->r.lanes; ++e) lengths_out[e] = c[(size_t)e] > 0 ? c[(size_t)e] - 1 : 0;
    return B200RL_OK;
}
/* length of lane 0 (lanes = 1 is the reference's single stream: 0 after the first state, 1 after the first transition) */
int b200rl_traj_length(b200rl_traj* t, int64_t* frames_out) {
    REQUIRE(t && frames_out, B200RL_ERR_INVALID, "null argument");
    TRY(ctx_bind(t->ctx));
    int32_t c = 0;
    CUDA_TRY(cudaMemcpyAsync(&c, t->r.count, 4, cudaMemcpyDeviceToHost, t->ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(t->ctx->stream));
    *frames_out = c > 0 ? c - 1 : 0;
    return B200RL_OK;
}
/* number of sampleable entries over all lanes (synchronises) */
int b200rl_traj_n_sampleable(b200rl_traj* t, int64_t* out) {
    REQUIRE(t && out, B200RL_ERR_INVALID, "null argument");
    TRY(ctx_bind(t->ctx));
    long long v = 0;
    CUDA_TRY(cudaMemcpyAsync(&v, t->r.n_valid, 8, cudaMemcpyDeviceToHost, t->ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(t->ctx->stream));
    *out = v;
    return B200RL_OK;
}

/* push!(trajectory, (state = s0,)) — the PreEpisodeStage push (agent_base.jl:45-47).  mode 0: every lane starts an episode
 * (forced reset); mode 1: only the lanes whose last transition was terminal (soft reset of a MultiThreadEnv-style batch). */
int b200rl_traj_push_episode_start(b200rl_traj* t, const float* obs, int on_device, int mode) {
    REQUIRE(t && obs && (mode == 0 || mode == 1), B200RL_ERR_INVALID, "bad argument");
    TRY(ctx_bind(t->ctx));
    const void* d = obs;
    if (!on_device) TRY(stage_in(t, obs, (size_t)t->r.ns * t->r.lanes * 4, 0, &d));
    push_episode_start_kernel<<<grid_for(t->r.lanes, 256), 256, 0, t->ctx->stream>>>(t->r, (const float*)d, mode, t->default_priority,
                                                                                     t->prioritized ? t->keys : nullptr, t->vals);
    LAUNCH_CHECK(t->ctx);
    TRY(tree_apply(t));
    if (!on_device) CUDA_TRY(cudaStreamSynchronize(t->ctx->stream));
    return B200RL_OK;
}
int b200rl_traj_push_state(b200rl_traj* t, const float* obs, int on_device) { return b200rl_traj_push_episode_start(t, obs, on_device, 0); }

int b200rl_traj_push(b200rl_traj* t, const int32_t* action, const float* reward, const uint8_t* terminal, const float* next_obs,
                     int on_device) {
    REQUIRE(t && action && reward && terminal && next_obs, B200RL_ERR_INVALID, "null argument");
    TRY(ctx_bind(t->ctx));
    Ring& r = t->r;
    const void *da = action, *dr = reward, *dt = terminal, *ds = next_obs;
    if (!on_device) {
        size_t L = (size_t)r.lanes;
        TRY(stage_in(t, next_obs, L * r.ns * 4, 0, &ds));
        TRY(stage_in(t, action, L * 4, L * r.ns * 4, &da));
        TRY(stage_in(t, reward, L * 4, L * r.ns * 4 + L * 4, &dr));
        TRY(stage_in(t, terminal, L, L * r.ns * 4 + L * 8, &dt));
    }
    push_sart_kernel<<<grid_for(r.lanes, 256), 256, 0, t->ctx->stream>>>(r, (const int32_t*)da, (const float*)dr, (const uint8_t*)dt, (const float*)ds,
                                                                            t->default_priority, t->prioritized ? t->keys : nullptr, t->vals);
    LAUNCH_CHECK(t->ctx);
    TRY(tree_apply(t));
    t->pushed += 1;
    if (!on_device) CUDA_TRY(cudaStreamSynchronize(t->ctx->stream));
    return B200RL_OK;
}

/* BatchSampler / prioritised sampler + gather into the trajectory's device batch buffers */
int b200rl_traj_sample(b200rl_traj* t, float beta) {
    REQUIRE(t && t->B > 0, B200RL_ERR_INVALID, "trajectory was created without a sampler");
    REQUIRE(t->pushed >= 1, B200RL_ERR_INVALID, "nothing to sample yet");
    TRY(ctx_bind(t->ctx));
    if (t->prioritized) {
        sample_gather_kernel<true><<<grid_for(t->B, 128), 128, 0, t->ctx->stream>>>(t->r, t->slots, t->B, beta, t->batch);
        LAUNCH_CHECK(t->ctx);
        normalize_weights_kernel<<<1, 1024, 0, t->ctx->stream>>>(t->batch.w, t->B);
        LAUNCH_CHECK(t->ctx);
    } else {
        sample_gather_kernel<false><<<grid_for(t->B, 128), 128, 0, t->ctx->stream>>>(t->r, t->slots, t->B, beta, t->batch);
        LAUNCH_CHECK(t->ctx);
    }
    return B200RL_OK;
}

/* Checkpoint of the ring (docs/src/How_to_use_hooks.md:124-167 pattern): field 0 state (ns, lanes, cap+1) f32 | 1 action i32 |
 * 2 reward f32 | 3 flag u8 (bit0 terminal, bit1 sampleable) | 4 head (lanes) i32 | 5 count (lanes) i32 | 6 pending (lanes) u8 |
 * 7 n_sampleable i64 | 8 sum tree (2L) f32 | 9 sampler streams (4, B) u64.  bytes_out (may be NULL) receives the field size. */
static int traj_field(b200rl_traj* t, int field, void** p, size_t* bytes) {
    const size_t slots = (size_t)t->r.lanes * (size_t)(t->r.cap + 1), L = (size_t)t->r.lanes;
    switch (field) {
        case 0: *p = t->r.state; *bytes = slots * t->r.ns * 4; return B200RL_OK;
        case 1: *p = t->r.action; *bytes = slots * 4; return B200RL_OK;
        case 2: *p = t->r.reward; *bytes = slots * 4; return B200RL_OK;
        case 3: *p = t->r.flag; *bytes = slots; return B200RL_OK;
        case 4: *p = t->r.head; *bytes = L * 4; return B200RL_OK;
        case 5: *p = t->r.count; *bytes = L * 4; return B200RL_OK;
        case 6: *p = t->r.pending; *bytes = L; return B200RL_OK;
        case 7: *p = t->r.n_valid; *bytes = 8; return B200RL_OK;
        case 8: REQUIRE(t->prioritized, B200RL_ERR_INVALID, "no sum tree"); *p = t->r.tree; *bytes = (size_t)(2 * t->r.L) * 4; return B200RL_OK;
        case 9: REQUIRE(t->B > 0, B200RL_ERR_INVALID, "no sampler"); *p = t->slots; *bytes = (size_t)t->B * 32; return B200RL_OK;
    }
    REQUIRE(false, B200RL_ERR_INVALID, "unknown trajectory field");
}
int b200rl_traj_field_bytes(b200rl_traj* t, int field, size_t* bytes_out) {
    REQUIRE(t && bytes_out, B200RL_ERR_INVALID, "null argument");
    void* p;
    return traj_field(t, field, &p, bytes_out);
}
int b200rl_traj_get(b200rl_traj* t, int field, void* host_dst, size_t bytes) {
    REQUIRE(t && host_dst, B200RL_ERR_INVALID, "null argument");
    TRY(ctx_bind(t->ctx));
    void* p; size_t need;
    TRY(traj_field(t, field, &p, &need));
    REQUIRE(bytes >= need, B200RL_ERR_INVALID, "destination too small");
    CUDA_TRY(cudaMemcpyAsync(host_dst, p, need, cudaMemcpyDeviceToHost, t->ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(t->ctx->stream));
    return B200RL_OK;
}
int b200rl_traj_set(b200rl_traj* t, int field, const void* host_src, size_t bytes) {
    REQUIRE(t && host_src, B200RL_ERR_INVALID, "null argument");
    TRY(ctx_bind(t->ctx));
    void* p; size_t need;
    TRY(traj_field(t, field, &p, &need));
    REQUIRE(bytes >= need, B200RL_ERR_INVALID, "source too small");
    CUDA_TRY(cudaMemcpyAsync(p, host_src, need, cudaMemcpyHostToDevice, t->ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(t->ctx->stream));
    if (field == 5) t->pushed = 1;   // a restored ring may be sampled
    return B200RL_OK;
}
/* field: 0 state (ns,B) 1 action (B) i32 2 reward 3 terminal u8 4 next_state 5 key i64 6 priority 7 weight 8 sampler rng (4,B) */
int b200rl_traj_batch_get(b200rl_traj* t, int field, void* host_dst, size_t bytes) {
    REQUIRE(t && host_dst && t->B > 0, B200RL_ERR_INVALID, "bad argument");
    TRY(ctx_bind(t->ctx));
    size_t B = (size_t)t->B;
    const void* src = nullptr;
    size_t need = 0;
    switch (field) {
        case 0: src = t->batch.s; need = B * t->r.ns * 4; break;
        case 1: src = t->batch.a; need = B * 4; break;
        case 2: src = t->batch.r; need = B * 4; break;
        case 3: src = t->batch.t; need = B; break;
        case 4: src = t->batch.s2; need = B * t->r.ns * 4; break;
        case 5: src = t->batch.key; need = B * 8; break;
        case 6: src = t->batch.prio; need = B * 4; break;
        case 7: src = t->batch.w; need = B * 4; break;
        case 8: src = t->slots; need = B * 32; break;
        default: REQUIRE(false, B200RL_ERR_INVALID, "unknown batch field");
    }
    REQUIRE(bytes >= need, B200RL_ERR_INVALID, "destination too small");
    CUDA_TRY(cudaMemcpyAsync(host_dst, src, need, cudaMemcpyDeviceToHost, t->ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(t->ctx->stream));
    return B200RL_OK;
}

/* priority write-back for the keys of the last sampled batch */
int b200rl_traj_update_priority(b200rl_traj* t, const float* prio, int on_device) {
    REQUIRE(t && prio && t->prioritized && t->B > 0, B200RL_ERR_INVALID, "bad argument");
    TRY(ctx_bind(t->ctx));
    const float* d = prio;
    if (!on_device) {
        CUDA_TRY(cudaMemcpyAsync(t->new_prio, prio, (size_t)t->B * 4, cudaMemcpyHostToDevice, t->ctx->stream));
        d = t->new_prio;
    }
    tree_update_keys_kernel<<<1, 1024, 0, t->ctx->stream>>>(t->r.tree, t->r.L, t->batch.key, d, t->B);
    LAUNCH_CHECK(t->ctx);
    if (!on_device) CUDA_TRY(cudaStreamSynchronize(t->ctx->stream));
    return B200RL_OK;
}

int b200rl_traj_total_priority(b200rl_traj* t, float* out) {
    REQUIRE(t && out && t->prioritized, B200RL_ERR_INVALID, "bad argument");
    TRY(ctx_bind(t->ctx));
    CUDA_TRY(cudaMemcpyAsync(out, t->r.tree + 1, 4, cudaMemcpyDeviceToHost, t->ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(t->ctx->stream));
    return B200RL_OK;
}

}  // extern "C"

// ---- internal accessors for algo.cu -----------------------------------------------------------
TrajBatchView b200rl_traj_internal_batch(b200rl_traj* t) {
    return TrajBatchView{t->batch.s, t->batch.a, t->batch.r, t->batch.t, t->batch.s2, t->prioritized ? t->batch.w : nullptr, t->B, t->r.ns};
}
bool b200rl_traj_internal_prioritized(b200rl_traj* t) { return t->prioritized; }
b200rl_ctx* b200rl_traj_internal_ctx(b200rl_traj* t) { return t->ctx; }
int64_t b200rl_traj_internal_lanes(b200rl_traj* t) { return t->r.lanes; }
int b200rl_traj_internal_priority_from_td(b200rl_traj* t, const float* td_dev, float eps, float alpha) {
    td_to_priority_kernel<<<grid_for(t->B, 256), 256, 0, t->ctx->stream>>>(td_dev, t->new_prio, t->B, eps, alpha);
    LAUNCH_CHECK(t->ctx);
    tree_update_keys_kernel<<<1, 1024, 0, t->ctx->stream>>>(t->r.tree, t->r.L, t->batch.key, t->new_prio, t->B);
    LAUNCH_CHECK(t->ctx);
    return B200RL_OK;
}
