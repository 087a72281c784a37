// algo.cu — host-side orchestration behind the C ABI: network handle (FluxApproximator +
// optimiser state + TargetNetwork), the on-policy agent (PPO / A2C: plan! -> act! -> push! ->
// optimise!), and the DQN update on a prioritised trajectory.  All arithmetic is in the
// kernels of nn.cu / returns.cu / traj.cu / env.cu; this file sequences launches on the ctx
// stream and owns the rollout tensors.
//
// Reference anchors: Agent stage pushes RLCore/src/policies/agent/agent_base.jl:45-66;
// FluxApproximator/optimise! policies/learners/flux_approximator.jl:11-46; TargetNetwork
// target_network.jl:27-88; PPO/A2C/DQN update rules: ReinforcementLearningZoo (absent from the
// snapshot; SURVEY Appendix B), hyper-parameters docs/homepage/blog/a_practical_introduction_to_RL.jl/index.html:15238-15286.
#include "internal.h"
#include "nn.cuh"
#include "opt_path.h"

static bool fused_rollout_enabled() {   // B200RL_FUSED_ROLLOUT=0: step through plan!/act! launches instead (same results)
    static int v = -1;
    if (v < 0) { const char* e = getenv("B200RL_FUSED_ROLLOUT"); v = (e && e[0] == '0') ? 0 : 1; }
    return v != 0;
}

namespace {
__global__ void clamp_copy_kernel(float* __restrict__ dst, const float* __restrict__ src, int64_t n, float lo, float hi) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = fminf(fmaxf(src[i], lo), hi);
}
__global__ void copy_f32_kernel(float* __restrict__ dst, const float* __restrict__ src, int64_t n) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = src[i];
}
__global__ void stats_row_kernel(float* __restrict__ row, const float* __restrict__ loss4, const float* __restrict__ gnorm,
                                 unsigned int* __restrict__ tick) {
    if (threadIdx.x < 4) row[threadIdx.x] = loss4[threadIdx.x];
    if (threadIdx.x == 4) row[4] = *gnorm;
    if (threadIdx.x == 5 && tick) *tick += 1u;
}
// After GAE: one 32-byte record per rollout sample {state (zero padded to 4), action bits, logp_old, advantage, return}, so the
// randomly permuted minibatch gather of K7 touches ONE DRAM sector per sample instead of one per array (5 arrays: ~4x the
// algorithmic bytes, profiles/r01_ncu_summary.md).  Streaming: 32 B read + 32 B written per sample, fully coalesced.
template <int NS>
__global__ void __launch_bounds__(256) pack_records_kernel(float4* __restrict__ rec, const float* __restrict__ states, const uint32_t* __restrict__ actions,
                                                          const float* __restrict__ logp, const float* __restrict__ adv, const float* __restrict__ ret,
                                                          int64_t total) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= total) return;
    float4 st = make_float4(0.f, 0.f, 0.f, 0.f);
    if (NS == 4) st = reinterpret_cast<const float4*>(states)[j];
    else {
        float x[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int i = 0; i < NS; ++i) x[i] = states[(int64_t)NS * j + i];
        st = make_float4(x[0], x[1], x[2], x[3]);
    }
    float4 sc = make_float4(__uint_as_float(actions[j]), logp[j], adv[j], ret[j]);
    // 32 lanes x 32 B = 1 KB contiguous per warp: two 16-byte stores per thread land in the same sector
    rec[2 * j] = st;
    rec[2 * j + 1] = sc;
}
__global__ void sum_norm_partials_kernel(const double* __restrict__ partials, int n, double* __restrict__ out2) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        double a = 0, b = 0;
        for (int k = 0; k < n; ++k) { a += partials[2 * k]; b += partials[2 * k + 1]; }
        out2[0] = a; out2[1] = b;
    }
}
__global__ void finalize_norm2_kernel(const double* __restrict__ sums2, double count, float* __restrict__ out2) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        double mean = sums2[0] / count;
        double var = (sums2[1] - count * mean * mean) / (count - 1.0);
        if (var < 0) var = 0;
        float sd = (float)sqrt(var);
        sd = sd < 1e-8f ? 1e-8f : (sd > 1000.0f ? 1000.0f : sd);
        out2[0] = (float)mean;
        out2[1] = 1.0f / sd;
    }
}
}  // namespace

// ------------------------------------------------------------------ network handle ---------
struct b200rl_net {
    b200rl_ctx* ctx;
    int kind;  // 0 actor-critic categorical, 1 actor-critic gaussian, 2 Q-network
    MlpDesc actor, critic;
    int64_t np;
    float *params, *grad, *m, *v, *beta_t, *target;
    float* partial; int n_partials;
    float* loss_partial; float* loss4; float* gnorm;
    double* cta_sumsq; unsigned int* counter2;
    float lr, b1, b2, eps, max_grad_norm;
    uint64_t n_updates;
};

static int make_descs(const b200rl_net_desc* d, MlpDesc* actor, MlpDesc* critic) {
    REQUIRE(d, B200RL_ERR_INVALID, "null desc");
    REQUIRE(d->kind >= 0 && d->kind <= 2, B200RL_ERR_INVALID, "kind must be 0 (actor-critic categorical), 1 (gaussian) or 2 (Q-network)");
    REQUIRE(d->n_in >= 1 && d->n_in <= kInMax, B200RL_ERR_UNSUPPORTED, "n_in must be 1..4");
    REQUIRE(d->hidden == 64 || d->hidden == 128, B200RL_ERR_UNSUPPORTED, "hidden must be 64 or 128");
    REQUIRE(d->act == 0 || d->act == 1, B200RL_ERR_INVALID, "act must be 0 (relu) or 1 (tanh)");
    if (d->kind == 1) REQUIRE(d->n_out == 1, B200RL_ERR_UNSUPPORTED, "gaussian policy supports a 1-d action");
    else REQUIRE(d->n_out >= 1 && d->n_out <= kOutMax, B200RL_ERR_UNSUPPORTED, "n_out must be 1..4");
    *actor = MlpDesc{d->n_in, d->hidden, d->act, d->kind == 1 ? 2 : d->n_out, d->kind == 1 ? 1 : 0};
    *critic = MlpDesc{d->n_in, d->hidden, d->act, 1, 0};
    return B200RL_OK;
}

static AcHyper hyper_of(const b200rl_onpolicy_config& c) {
    return AcHyper{c.clip_range, c.w_actor, c.w_critic, c.w_entropy, c.min_sigma, c.max_sigma, c.normalize_advantage, c.algo};
}

// rows {4 loss sums, grad norm} (stride 8) -> {actor_loss, critic_loss, entropy, loss, grad_norm, 0} (stride 6), losses = sums * invB
static void decode_stats_rows(const b200rl_onpolicy_config& c, const float* rows, int n_rows, float invB, float* out) {
    for (int r = 0; r < n_rows; ++r) {
        const float* s = rows + (size_t)r * 8;
        float* o = out + (size_t)r * 6;
        o[0] = s[0] * invB; o[1] = s[2] * invB; o[2] = s[1] * invB;
        o[3] = c.w_actor * o[0] + c.w_critic * o[1] - c.w_entropy * o[2];
        o[4] = s[4]; o[5] = 0.f;
    }
}

// Which kernels run the optimiser step of `n` (opt_path.h).  fused: the caller can run the step in the tail of its tensor-core loss +
// backward launch on a minibatch of B samples.
static OptPath net_opt_path(const b200rl_net* n, bool fused, const AcHyper& hp, int64_t B) {
    b200rl_ctx* ctx = n->ctx;
    P2PTable peers = {};
    OptPathIn in;
    in.world = b200rl_comm_world(ctx);
    in.p2p = b200rl_comm_p2p_table(ctx, &peers);
    in.exclusive = peers.exclusive != 0;
    in.fused_step = fused && nn_fused_step_enabled();
    in.tc_bwd = nn_tc_enabled() && nn_tc_bwd_supported(n->actor, n->critic);
    in.tail_fits = in.fused_step && in.tc_bwd && nn_tc_fused_tail_fits(ctx, n->actor, hp, B, n->np);
    in.fits_inbox = (size_t)n->np + 4 <= kP2PXCap;
    in.coresident = (int)grid_for(n->np, 256) <= ctx->sm_count;
    return opt_path(in);
}

// The optimiser state of `n` with the step's hyper-parameters (Cfg: b200rl_onpolicy_config or b200rl_dqn_config).  stats_row (may be
// null) receives {4 loss sums, grad norm}; tick (may be null) is a device counter the step increments once.
template <class Cfg>
static OptStep net_opt_state(const b200rl_net* n, const Cfg& c, float lr, float* stats_row, unsigned int* tick) {
    OptStep s = {};
    s.params = n->params; s.grad = n->grad; s.m = n->m; s.v = n->v; s.beta_t = n->beta_t;
    s.loss_out4 = n->loss4; s.stats_row = stats_row; s.gnorm_out = n->gnorm;
    s.cta_sumsq = n->cta_sumsq; s.counter = n->counter2; s.tick = tick;
    s.max_norm = c.max_grad_norm; s.lr = lr; s.b1 = c.beta1; s.b2 = c.beta2; s.eps = c.eps;
    if (b200rl_comm_p2p_table(n->ctx, &s.tab)) s.seq_ptr = b200rl_comm_p2p_seq_dev(n->ctx);
    return s;
}

// The optimiser step on the n_partials gradient rows / n_loss loss rows in n->partial / n->loss_partial, by every path but
// OPT_FUSED_TAIL (which runs inside the loss + backward launch, nn_ac_loss_grad_step).
static int net_opt_step(b200rl_net* n, OptPath path, int n_partials, int n_loss, const OptStep& st) {
    b200rl_ctx* ctx = n->ctx;
    if (path != OPT_NCCL_CHAIN) return nn_reduce_clip_adam(ctx, n->partial, n_partials, n->np, n->loss_partial, n_loss, st);
    TRY(nn_reduce_partials(ctx, n->partial, n_partials, n->np, st.grad, n->loss_partial, n_loss, st.loss_out4));
    if (b200rl_comm_world(ctx) > 1) {
        TRY(b200rl_comm_allreduce_internal(ctx, st.grad, n->np, 0));
        TRY(b200rl_comm_allreduce_internal(ctx, st.loss_out4, 4, 0));
    }
    TRY(nn_clip_adam(ctx, st.params, st.grad, st.m, st.v, st.beta_t, n->np, st.max_norm, st.lr, st.b1, st.b2, st.eps, 1.0f, st.gnorm_out));
    if (st.stats_row) {
        stats_row_kernel<<<1, 32, 0, ctx->stream>>>(st.stats_row, st.loss_out4, st.gnorm_out, st.tick);
        LAUNCH_CHECK(ctx);
    }
    return B200RL_OK;
}

extern "C" {

int b200rl_net_nparams(const b200rl_net_desc* d, int64_t* out) {
    MlpDesc a, c;
    TRY(make_descs(d, &a, &c));
    REQUIRE(out, B200RL_ERR_INVALID, "null out");
    *out = d->kind == 2 ? a.nparams() : a.nparams() + c.nparams();
    return B200RL_OK;
}

int b200rl_net_destroy(b200rl_net* n) {
    if (!n) return B200RL_OK;
    cudaSetDevice(n->ctx->device);
    cudaStreamSynchronize(n->ctx->stream);
    cudaFree(n->params); cudaFree(n->grad); cudaFree(n->m); cudaFree(n->v); cudaFree(n->beta_t); cudaFree(n->target);
    cudaFree(n->partial); cudaFree(n->loss_partial); cudaFree(n->loss4); cudaFree(n->gnorm); cudaFree(n->cta_sumsq); cudaFree(n->counter2);
    delete n;
    return B200RL_OK;
}

/* Replaces FluxApproximator(model, optimiser) (+ TargetNetwork for kind 2): takes the flat
 * Flux.destructure parameter vector; optimiser = Adam(1e-3, (0.9, 0.999), 1e-8), clip 0.5 until
 * b200rl_net_configure_optimizer is called. */
int b200rl_net_create(b200rl_ctx* ctx, const b200rl_net_desc* d, const float* params_host, b200rl_net** out) {
    TRY(ctx_bind(ctx));
    REQUIRE(out && params_host, B200RL_ERR_INVALID, "null argument");
    b200rl_net* n = new b200rl_net();
    memset(n, 0, sizeof *n);
    n->ctx = ctx; n->kind = d ? d->kind : 0;
    int s = make_descs(d, &n->actor, &n->critic);
    if (s != B200RL_OK) { delete n; return s; }
    n->np = n->kind == 2 ? n->actor.nparams() : n->actor.nparams() + n->critic.nparams();
    n->lr = 1e-3f; n->b1 = 0.9f; n->b2 = 0.999f; n->eps = 1e-8f; n->max_grad_norm = 0.5f;
    size_t bytes = (size_t)n->np * sizeof(float);
    n->n_partials = n->kind == 2 ? nn_dqn_max_partials(ctx, n->actor.H) : nn_grid_ctas(ctx, n->actor.H);
    int n_loss_rows = 2 * (n->n_partials > ctx->sm_count ? n->n_partials : ctx->sm_count);
#define NET_TRY(x) do { cudaError_t _e = (x); if (_e != cudaSuccess) { b200rl_set_error("%s -> %s", #x, cudaGetErrorString(_e)); b200rl_net_destroy(n); return B200RL_ERR_CUDA; } } while (0)
    NET_TRY(cudaMalloc(&n->params, bytes)); NET_TRY(cudaMalloc(&n->grad, bytes)); NET_TRY(cudaMalloc(&n->m, bytes)); NET_TRY(cudaMalloc(&n->v, bytes));
    NET_TRY(cudaMalloc(&n->beta_t, 2 * sizeof(float)));
    if (n->kind == 2) NET_TRY(cudaMalloc(&n->target, bytes));
    NET_TRY(cudaMalloc(&n->partial, (size_t)n->n_partials * bytes));
    NET_TRY(cudaMalloc(&n->loss_partial, (size_t)n_loss_rows * 4 * sizeof(float)));
    NET_TRY(cudaMalloc(&n->loss4, 4 * sizeof(float))); NET_TRY(cudaMalloc(&n->gnorm, sizeof(float)));
    NET_TRY(cudaMalloc(&n->cta_sumsq, 256 * sizeof(double))); NET_TRY(cudaMalloc(&n->counter2, 4 * sizeof(unsigned int)));
    NET_TRY(cudaMemsetAsync(n->counter2, 0, 4 * sizeof(unsigned int), ctx->stream));
    NET_TRY(cudaMemcpyAsync(n->params, params_host, bytes, cudaMemcpyHostToDevice, ctx->stream));
    if (n->kind == 2) NET_TRY(cudaMemcpyAsync(n->target, params_host, bytes, cudaMemcpyHostToDevice, ctx->stream));
    NET_TRY(cudaMemsetAsync(n->grad, 0, bytes, ctx->stream)); NET_TRY(cudaMemsetAsync(n->m, 0, bytes, ctx->stream));
    NET_TRY(cudaMemsetAsync(n->v, 0, bytes, ctx->stream));
    NET_TRY(cudaMemsetAsync(n->partial, 0, (size_t)n->n_partials * bytes, ctx->stream));
    NET_TRY(cudaMemsetAsync(n->loss_partial, 0, (size_t)n_loss_rows * 4 * sizeof(float), ctx->stream));
    float bt[2] = {n->b1, n->b2};
    NET_TRY(cudaMemcpyAsync(n->beta_t, bt, sizeof bt, cudaMemcpyHostToDevice, ctx->stream));
    NET_TRY(cudaStreamSynchronize(ctx->stream));
#undef NET_TRY
    *out = n;
    return B200RL_OK;
}

int b200rl_net_configure_optimizer(b200rl_net* n, float lr, float beta1, float beta2, float eps, float max_grad_norm) {
    REQUIRE(n, B200RL_ERR_INVALID, "null net");
    TRY(ctx_bind(n->ctx));
    n->lr = lr; n->b1 = beta1; n->b2 = beta2; n->eps = eps; n->max_grad_norm = max_grad_norm;
    if (n->n_updates == 0) {
        float bt[2] = {beta1, beta2};
        CUDA_TRY(cudaMemcpyAsync(n->beta_t, bt, sizeof bt, cudaMemcpyHostToDevice, n->ctx->stream));
        CUDA_TRY(cudaStreamSynchronize(n->ctx->stream));
    }
    return B200RL_OK;
}

/* which: 0 params, 1 last (clipped) gradient, 2 Adam m, 3 Adam v, 4 beta_t (2 floats), 5 target params */
static int net_buf(b200rl_net* n, int which, float** p, int64_t* len) {
    switch (which) {
        case 0: *p = n->params; *len = n->np; return B200RL_OK;
        case 1: *p = n->grad; *len = n->np; return B200RL_OK;
        case 2: *p = n->m; *len = n->np; return B200RL_OK;
        case 3: *p = n->v; *len = n->np; return B200RL_OK;
        case 4: *p = n->beta_t; *len = 2; return B200RL_OK;
        case 5: REQUIRE(n->target, B200RL_ERR_INVALID, "no target network"); *p = n->target; *len = n->np; return B200RL_OK;
    }
    REQUIRE(false, B200RL_ERR_INVALID, "unknown buffer id");
}
/* export / import of parameters and optimiser state (checkpoint hook pattern, docs/src/How_to_use_hooks.md:124-167) */
int b200rl_net_get(b200rl_net* n, int which, float* host_dst, int64_t count) {
    REQUIRE(n && host_dst, B200RL_ERR_INVALID, "null argument");
    TRY(ctx_bind(n->ctx));
    float* p; int64_t len;
    TRY(net_buf(n, which, &p, &len));
    REQUIRE(count >= len, B200RL_ERR_INVALID, "destination too small");
    CUDA_TRY(cudaMemcpyAsync(host_dst, p, (size_t)len * 4, cudaMemcpyDeviceToHost, n->ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(n->ctx->stream));
    return B200RL_OK;
}
int b200rl_net_set(b200rl_net* n, int which, const float* host_src, int64_t count) {
    REQUIRE(n && host_src, B200RL_ERR_INVALID, "null argument");
    TRY(ctx_bind(n->ctx));
    float* p; int64_t len;
    TRY(net_buf(n, which, &p, &len));
    REQUIRE(count >= len, B200RL_ERR_INVALID, "source too small");
    CUDA_TRY(cudaMemcpyAsync(p, host_src, (size_t)len * 4, cudaMemcpyHostToDevice, n->ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(n->ctx->stream));
    return B200RL_OK;
}
int b200rl_net_ptr(b200rl_net* n, int which, void** dptr_out) {
    REQUIRE(n && dptr_out, B200RL_ERR_INVALID, "null argument");
    float* p; int64_t len;
    TRY(net_buf(n, which, &p, &len));
    *dptr_out = p;
    return B200RL_OK;
}

/* optimiser steps taken so far (drives the TargetNetwork's sync_freq phase, target_network.jl:70-88; part of a checkpoint) */
int b200rl_net_get_step(b200rl_net* n, int64_t* out) {
    REQUIRE(n && out, B200RL_ERR_INVALID, "null argument");
    *out = (int64_t)n->n_updates;
    return B200RL_OK;
}
int b200rl_net_set_step(b200rl_net* n, int64_t step) {
    REQUIRE(n && step >= 0, B200RL_ERR_INVALID, "bad argument");
    n->n_updates = (uint64_t)step;
    return B200RL_OK;
}
/* TargetNetwork sync: target = rho*target + (1-rho)*model (rho = 0: hard copy) — target_network.jl:70-88 */
int b200rl_net_target_sync(b200rl_net* n, float rho) {
    REQUIRE(n && n->target, B200RL_ERR_INVALID, "no target network");
    TRY(ctx_bind(n->ctx));
    return nn_target_sync(n->ctx, n->target, n->params, n->np, rho);
}

static int stage_obs(b200rl_net* n, const float* obs, int64_t N, int on_device, const float** dev, size_t extra, void** extra_dev) {
    size_t ob = (size_t)N * n->actor.in * 4;
    if (on_device && extra == 0) { *dev = obs; return B200RL_OK; }
    void* s;
    TRY(ctx_scratch(n->ctx, ob + extra + 512, &s));
    if (!on_device) { CUDA_TRY(cudaMemcpyAsync(s, obs, ob, cudaMemcpyHostToDevice, n->ctx->stream)); *dev = (const float*)s; }
    else *dev = obs;
    if (extra_dev) *extra_dev = (char*)s + ((ob + 255) / 256) * 256;
    return B200RL_OK;
}

/* plan!(policy, env) for a batch of observations (in, N): action (int32 1-based | float), log-prob and V(s).
 * rng = (4, N) uint64 DEVICE policy streams (advanced in place).  Outputs may be NULL.  on_device applies to obs and outputs. */
int b200rl_net_act(b200rl_net* n, const float* obs, int64_t N, uint64_t* rng_dev, void* action_out, float* logp_out, float* value_out,
                   float* heads_out, int on_device) {
    REQUIRE(n && obs && rng_dev && n->kind != 2, B200RL_ERR_INVALID, "bad argument (actor-critic nets only)");
    TRY(ctx_bind(n->ctx));
    AcHyper hp{0.1f, 1.f, 0.5f, 0.001f, 0.f, __builtin_inff(), 0, 0};
    const float* dobs;
    size_t ho = (size_t)N * n->actor.nout * 4;
    void* ex = nullptr;
    TRY(stage_obs(n, obs, N, on_device, &dobs, on_device ? 0 : (size_t)N * 12 + ho + 1024, &ex));
    if (on_device)
        return nn_policy_act(n->ctx, n->actor, n->critic, n->params, hp, dobs, N, (unsigned long long*)rng_dev, action_out, logp_out, value_out,
                             heads_out, nullptr);
    float* da = (float*)ex; float* dl = da + N; float* dv = dl + N; float* dh = dv + N;
    TRY(nn_policy_act(n->ctx, n->actor, n->critic, n->params, hp, dobs, N, (unsigned long long*)rng_dev, da, dl, dv, heads_out ? dh : nullptr, nullptr));
    if (action_out) CUDA_TRY(cudaMemcpyAsync(action_out, da, (size_t)N * 4, cudaMemcpyDeviceToHost, n->ctx->stream));
    if (logp_out) CUDA_TRY(cudaMemcpyAsync(logp_out, dl, (size_t)N * 4, cudaMemcpyDeviceToHost, n->ctx->stream));
    if (value_out) CUDA_TRY(cudaMemcpyAsync(value_out, dv, (size_t)N * 4, cudaMemcpyDeviceToHost, n->ctx->stream));
    if (heads_out) CUDA_TRY(cudaMemcpyAsync(heads_out, dh, ho, cudaMemcpyDeviceToHost, n->ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(n->ctx->stream));
    return B200RL_OK;
}

/* critic V(s) (kinds 0/1: out (N)) or Q(s, .) (kind 2: out (n_out, N)); use_target selects the target network */
int b200rl_net_values(b200rl_net* n, const float* obs, int64_t N, float* out, int use_target, int on_device) {
    REQUIRE(n && obs && out, B200RL_ERR_INVALID, "null argument");
    TRY(ctx_bind(n->ctx));
    const MlpDesc& d = n->kind == 2 ? n->actor : n->critic;
    const float* p = n->kind == 2 ? (use_target ? n->target : n->params) : n->params + n->actor.nparams();
    REQUIRE(p, B200RL_ERR_INVALID, "no target network");
    const float* dobs;
    size_t ob = (size_t)N * d.nout * 4;
    void* ex = nullptr;
    TRY(stage_obs(n, obs, N, on_device, &dobs, on_device ? 0 : ob + 256, &ex));
    if (on_device) return nn_mlp_forward(n->ctx, d, p, dobs, N, out);
    TRY(nn_mlp_forward(n->ctx, d, p, dobs, N, (float*)ex));
    CUDA_TRY(cudaMemcpyAsync(out, ex, ob, cudaMemcpyDeviceToHost, n->ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(n->ctx->stream));
    return B200RL_OK;
}

/* epsilon-greedy action selection on Q(s, .) (EpsilonGreedyExplorer / QBasedPolicy plan!); all pointers DEVICE */
int b200rl_net_q_act(b200rl_net* n, const float* obs_dev, int64_t N, uint64_t* rng_dev, float epsilon, int32_t* action_out_dev) {
    REQUIRE(n && obs_dev && action_out_dev && n->kind == 2, B200RL_ERR_INVALID, "bad argument (Q-network only)");
    REQUIRE(epsilon <= 0.f || rng_dev, B200RL_ERR_INVALID, "rng required for epsilon > 0");
    TRY(ctx_bind(n->ctx));
    void* s;
    TRY(ctx_scratch(n->ctx, (size_t)N * n->actor.nout * 4 + 256, &s));
    return nn_q_act(n->ctx, n->actor, n->params, obs_dev, N, (unsigned long long*)rng_dev, epsilon, action_out_dev, (float*)s);
}

/* BatchExplorer(EpsilonGreedyExplorer) with the decay schedule evaluated per column on the device; all pointers DEVICE */
int b200rl_net_q_explore(b200rl_net* n, const float* obs_dev, int64_t N, uint64_t* rng_dev, const b200rl_explorer* ex, int32_t* action_out_dev) {
    REQUIRE(n && obs_dev && action_out_dev && rng_dev && ex && n->kind == 2, B200RL_ERR_INVALID, "bad argument (Q-network only)");
    REQUIRE(N > 0, B200RL_ERR_INVALID, "empty batch");
    REQUIRE((ex->kind == 0 || ex->kind == 1) && ex->warmup_steps >= 0 && ex->decay_steps >= 0, B200RL_ERR_INVALID, "bad explorer schedule");
    REQUIRE(ex->eps_stable >= 0.0 && ex->eps_stable <= 1.0 && ex->eps_init >= 0.0 && ex->eps_init <= 1.0, B200RL_ERR_INVALID, "epsilon outside [0, 1]");
    TRY(ctx_bind(n->ctx));
    void* s;
    TRY(ctx_scratch(n->ctx, (size_t)N * n->actor.nout * 4 + 256, &s));
    return nn_q_explore(n->ctx, n->actor, n->params, obs_dev, N, (unsigned long long*)rng_dev, *ex, action_out_dev, (float*)s);
}

/* One optimiser step from explicit on-policy minibatch arrays (all HOST; test / generic entry):
 * loss + gradient (K7), global-norm clip + Adam (K8).  losses_out[6] = actor_loss, critic_loss,
 * entropy, loss, grad_norm (pre-clip), 0.  apply_update = 0 leaves the parameters untouched (gradient only). */
int b200rl_net_ac_step(b200rl_net* n, const b200rl_onpolicy_config* cfg, const float* states, const void* actions, const float* logp_old,
                       const float* adv, const float* ret, int64_t total, const int32_t* idx, int64_t B, float adv_mean, float adv_inv_std,
                       int apply_update, float* losses_out) {
    REQUIRE(n && cfg && states && actions && adv && ret && n->kind != 2, B200RL_ERR_INVALID, "bad argument");
    TRY(ctx_bind(n->ctx));
    b200rl_ctx* ctx = n->ctx;
    int ns = n->actor.in;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
    const int64_t Beff = idx ? B : total;
    size_t o_s = take((size_t)total * ns * 4), o_a = take((size_t)total * 4), o_l = take((size_t)total * 4), o_ad = take((size_t)total * 4),
           o_r = take((size_t)total * 4), o_i = take((size_t)Beff * 4), o_n = take(8);
    void* sc;
    TRY(ctx_scratch(ctx, off, &sc));
    char* base = (char*)sc;
    std::vector<int32_t> iota;
    if (!idx) {  // identity order
        iota.resize((size_t)total);
        for (int64_t k = 0; k < total; ++k) iota[(size_t)k] = (int32_t)k;
        idx = iota.data();
    }
    CUDA_TRY(cudaMemcpyAsync(base + o_s, states, (size_t)total * ns * 4, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(base + o_a, actions, (size_t)total * 4, cudaMemcpyHostToDevice, ctx->stream));
    if (logp_old) CUDA_TRY(cudaMemcpyAsync(base + o_l, logp_old, (size_t)total * 4, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(base + o_ad, adv, (size_t)total * 4, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(base + o_r, ret, (size_t)total * 4, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(base + o_i, idx, (size_t)Beff * 4, cudaMemcpyHostToDevice, ctx->stream));
    float nm[2] = {adv_mean, adv_inv_std};
    CUDA_TRY(cudaMemcpyAsync(base + o_n, nm, 8, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));  // host buffers (incl. the local iota) are borrowed for this call only
    const AcHyper hp = hyper_of(*cfg);
    AcBatch b{(const float*)(base + o_s), ns, base + o_a, logp_old ? (const float*)(base + o_l) : nullptr, (const float*)(base + o_ad),
              (const float*)(base + o_r), (const int32_t*)(base + o_i), (uint32_t)total, 0u, 0u, nullptr, nullptr, Beff, 1.0f / (float)Beff,
              (const float*)(base + o_n)};
    int ctas = nn_ac_loss_grad(ctx, n->actor, n->critic, n->params, hp, b, n->partial, n->loss_partial);
    if (ctas < 0) return ctas;
    TRY(nn_reduce_partials(ctx, n->partial, ctas, n->np, n->grad, n->loss_partial, 2 * ctas, n->loss4));
    if (apply_update) {
        TRY(nn_clip_adam(ctx, n->params, n->grad, n->m, n->v, n->beta_t, n->np, cfg->max_grad_norm, cfg->lr, cfg->beta1, cfg->beta2, cfg->eps, 1.0f, n->gnorm));
        n->n_updates += 1;
    }
    if (losses_out) {
        float row[8] = {};   // {4 loss sums, grad norm}
        CUDA_TRY(cudaMemcpyAsync(row, n->loss4, 16, cudaMemcpyDeviceToHost, ctx->stream));
        if (apply_update) CUDA_TRY(cudaMemcpyAsync(row + 4, n->gnorm, 4, cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(cudaStreamSynchronize(ctx->stream));
        decode_stats_rows(*cfg, row, 1, 1.0f / (float)Beff, losses_out);
    }
    return B200RL_OK;
}

}  // extern "C"

// ------------------------------------------------------------------ on-policy agent --------
struct b200rl_onpolicy {
    b200rl_ctx* ctx;
    b200rl_net* net;
    b200rl_env* env;
    b200rl_onpolicy_config cfg;
    int64_t N;
    int T, t, ns;
    bool continuous;
    bool bootstrap_done;   // column T of states / values already written by the fused rollout
    unsigned long long* rng;
    float* states; void* actions; float* logp; float* rewards; uint8_t* terminals; float* values; float* adv; float* ret;
    float* act_clamped;
    double* norm_partials; double* norm_sums; float* norm2;
    int32_t* perm_dev;
    float* stats_dev; int stats_rows;
    float4* rec;                 // packed 32-byte records of the rollout (written after GAE, gathered by K7)
    unsigned int* upd_dev;       // device copy of n_updates: keys the minibatch permutation, ticked by the last optimiser step of an update
    uint64_t n_updates;
    // CUDA graph of one whole iteration (collect(T) + update) for b200rl_onpolicy_iterate
    cudaGraph_t graph; cudaGraphExec_t graph_exec; bool warmed; int graph_tc; uint64_t graph_env_gen; uint64_t graph_launches; int graph_failed;
};

static void* env_field(b200rl_env* e, int f) { void* p = nullptr; b200rl_env_ptr(e, f, &p); return p; }

static int64_t minibatch_size(const b200rl_onpolicy* a) { return a->N * a->T / a->cfg.n_microbatches; }   // per rank
static OptPath onpolicy_opt_path(const b200rl_onpolicy* a) { return net_opt_path(a->net, true, hyper_of(a->cfg), minibatch_size(a)); }
// the stats rows of the last update -> stats_host (n_epochs * n_microbatches, 6)
static int onpolicy_read_stats(b200rl_onpolicy* a, float* stats_host) {
    std::vector<float> tmp((size_t)a->stats_rows * 8);
    CUDA_TRY(cudaMemcpyAsync(tmp.data(), a->stats_dev, tmp.size() * 4, cudaMemcpyDeviceToHost, a->ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(a->ctx->stream));
    decode_stats_rows(a->cfg, tmp.data(), a->stats_rows, 1.0f / ((float)minibatch_size(a) * (float)b200rl_comm_world(a->ctx)), stats_host);
    return B200RL_OK;
}

extern "C" {

int b200rl_onpolicy_destroy(b200rl_onpolicy* a) {
    if (!a) return B200RL_OK;
    cudaSetDevice(a->ctx->device);
    cudaStreamSynchronize(a->ctx->stream);
    b200rl_env_internal_set_traj_targets(a->env, nullptr, nullptr);
    cudaFree(a->rng); cudaFree(a->states); cudaFree(a->actions); cudaFree(a->logp); cudaFree(a->rewards); cudaFree(a->terminals);
    cudaFree(a->values); cudaFree(a->adv); cudaFree(a->ret); cudaFree(a->act_clamped); cudaFree(a->norm_partials); cudaFree(a->norm_sums);
    cudaFree(a->norm2); cudaFree(a->perm_dev); cudaFree(a->stats_dev); cudaFree(a->rec); cudaFree(a->upd_dev);
    if (a->graph_exec) cudaGraphExecDestroy(a->graph_exec);
    if (a->graph) cudaGraphDestroy(a->graph);
    delete a;
    return B200RL_OK;
}

/* Agent(policy = PPOPolicy / A2CPolicy, trajectory = PPOTrajectory(capacity = update_freq)):
 * rollout tensors (N, T) env-fastest live on the device.  policy_rng: (4, N) host uint64, one
 * Xoshiro stream per env for action sampling (the reference draws a whole batch from one stream). */
int b200rl_onpolicy_create(b200rl_ctx* ctx, b200rl_net* net, b200rl_env* env, const b200rl_onpolicy_config* cfg, const uint64_t* policy_rng,
                           b200rl_onpolicy** out) {
    TRY(ctx_bind(ctx));
    REQUIRE(net && env && cfg && policy_rng && out, B200RL_ERR_INVALID, "null argument");
    REQUIRE(net->kind != 2, B200RL_ERR_INVALID, "needs an actor-critic network");
    REQUIRE(net->ctx == ctx && b200rl_env_internal_ctx(env) == ctx, B200RL_ERR_INVALID, "net/env belong to another ctx");
    REQUIRE(b200rl_env_internal_dtype(env) == B200RL_F32, B200RL_ERR_UNSUPPORTED, "the learners read Float32 observations: construct the env with T = Float32");
    REQUIRE(cfg->update_freq >= 1 && cfg->n_epochs >= 1 && cfg->n_microbatches >= 1, B200RL_ERR_INVALID, "bad config");
    int nobs = b200rl_env_internal_nobs(env);
    REQUIRE(nobs == net->actor.in, B200RL_ERR_INVALID, "network input width != observation width");
    bool cont = b200rl_env_internal_continuous(env);
    REQUIRE(cont == (net->kind == 1), B200RL_ERR_INVALID, "categorical policy needs a discrete env, gaussian a continuous one");
    int64_t N = b200rl_env_internal_n(env);
    REQUIRE((N * cfg->update_freq) % cfg->n_microbatches == 0, B200RL_ERR_INVALID, "N*T must be divisible by n_microbatches");
    REQUIRE(N * (int64_t)cfg->update_freq < (1ll << 31), B200RL_ERR_UNSUPPORTED, "rollout too large for 32-bit sample indices");
    b200rl_onpolicy* a = new b200rl_onpolicy();
    memset(a, 0, sizeof *a);
    a->ctx = ctx; a->net = net; a->env = env; a->cfg = *cfg; a->N = N; a->T = cfg->update_freq; a->t = 0; a->ns = nobs; a->continuous = cont;
    size_t NT_ = (size_t)N * a->T;
#define A_TRY(x) do { cudaError_t _e = (x); if (_e != cudaSuccess) { b200rl_set_error("%s -> %s", #x, cudaGetErrorString(_e)); b200rl_onpolicy_destroy(a); return _e == cudaErrorMemoryAllocation ? B200RL_ERR_OOM : B200RL_ERR_CUDA; } } while (0)
    A_TRY(cudaMalloc(&a->rng, (size_t)N * 32));
    A_TRY(cudaMalloc(&a->states, (size_t)N * nobs * (a->T + 1) * 4));
    A_TRY(cudaMalloc(&a->actions, NT_ * 4)); A_TRY(cudaMalloc(&a->logp, NT_ * 4)); A_TRY(cudaMalloc(&a->rewards, NT_ * 4));
    A_TRY(cudaMalloc(&a->terminals, NT_)); A_TRY(cudaMalloc(&a->values, (size_t)N * (a->T + 1) * 4));
    A_TRY(cudaMalloc(&a->adv, NT_ * 4)); A_TRY(cudaMalloc(&a->ret, NT_ * 4));
    A_TRY(cudaMalloc(&a->act_clamped, (size_t)N * 4));
    A_TRY(cudaMalloc(&a->norm_partials, (size_t)b200rl_gae_fused_partials_count(N) * sizeof(double)));
    A_TRY(cudaMalloc(&a->norm_sums, 2 * sizeof(double))); A_TRY(cudaMalloc(&a->norm2, 2 * sizeof(float)));
    a->stats_rows = cfg->n_epochs * cfg->n_microbatches;
    A_TRY(cudaMalloc(&a->stats_dev, (size_t)a->stats_rows * 8 * sizeof(float)));
    // staging for host-supplied shuffle!() results; allocated here because a device allocation inside update would
    // synchronise the device (and with it another rank of the same process that is waiting in the peer exchange)
    A_TRY(cudaMalloc(&a->perm_dev, (size_t)a->cfg.n_epochs * NT_ * 4));
    A_TRY(cudaMalloc(&a->rec, NT_ * 32));
    A_TRY(cudaMalloc(&a->upd_dev, sizeof(unsigned int)));
    A_TRY(cudaMemsetAsync(a->upd_dev, 0, sizeof(unsigned int), ctx->stream));
    A_TRY(cudaMemsetAsync(a->stats_dev, 0, (size_t)a->stats_rows * 8 * sizeof(float), ctx->stream));
    A_TRY(cudaMemcpyAsync(a->rng, policy_rng, (size_t)N * 32, cudaMemcpyHostToDevice, ctx->stream));
    A_TRY(cudaStreamSynchronize(ctx->stream));
#undef A_TRY
    TRY(b200rl_net_configure_optimizer(net, cfg->lr, cfg->beta1, cfg->beta2, cfg->eps, cfg->max_grad_norm));
    *out = a;
    return B200RL_OK;
}

/* RLBase.plan!(agent, env) + push!(agent, PreActStage): K6 on the env's current observation;
 * stores state / log-prob / V(s) into column t of the rollout and arms the env so that the
 * next act! writes reward / terminal into the same column.  actions_host (N) may be NULL. */
int b200rl_onpolicy_plan(b200rl_onpolicy* a, void* actions_host) {
    REQUIRE(a, B200RL_ERR_INVALID, "null agent");
    REQUIRE(a->t < a->T, B200RL_ERR_INVALID, "rollout is full: call b200rl_onpolicy_update first");
    TRY(ctx_bind(a->ctx));
    a->bootstrap_done = false;
    int64_t N = a->N;
    const float* obs = (const float*)env_field(a->env, B200RL_FIELD_OBS);
    const AcHyper hp = hyper_of(a->cfg);
    char* act_col = (char*)a->actions + (size_t)N * a->t * 4;
    TRY(nn_policy_act(a->ctx, a->net->actor, a->net->critic, a->net->params, hp, obs, N, a->rng, act_col, a->logp + (size_t)N * a->t,
                      a->values + (size_t)N * a->t, nullptr, a->states + (size_t)N * a->ns * a->t));
    TRY(b200rl_env_internal_set_traj_targets(a->env, a->rewards + (size_t)N * a->t, a->terminals + (size_t)N * a->t));
    if (actions_host) {
        CUDA_TRY(cudaMemcpyAsync(actions_host, act_col, (size_t)N * 4, cudaMemcpyDeviceToHost, a->ctx->stream));
        CUDA_TRY(cudaStreamSynchronize(a->ctx->stream));
    }
    return B200RL_OK;
}
/* RLBase.act!(env, planned action) device-to-device (auto-reset fused) */
int b200rl_onpolicy_act(b200rl_onpolicy* a) {
    REQUIRE(a, B200RL_ERR_INVALID, "null agent");
    TRY(ctx_bind(a->ctx));
    char* act_col = (char*)a->actions + (size_t)a->N * a->t * 4;
    if (a->continuous) {  // the env asserts a in -2.0..2.0; the stored (unclamped) action keeps its log-prob
        const float bound = b200rl_env_internal_kind(a->env) == B200RL_ENV_PENDULUM ? 2.0f : 1.0f;   // action_space -2.0..2.0 | -1.0..1.0
        clamp_copy_kernel<<<grid_for(a->N, 256), 256, 0, a->ctx->stream>>>(a->act_clamped, (const float*)act_col, a->N, -bound, bound);
        LAUNCH_CHECK(a->ctx);
        return b200rl_env_step(a->env, a->act_clamped, 1, 1);
    }
    return b200rl_env_step(a->env, act_col, 1, 1);
}
/* push!(agent, PostActStage, env, action): the transition of column t is complete */
int b200rl_onpolicy_push(b200rl_onpolicy* a) {
    REQUIRE(a, B200RL_ERR_INVALID, "null agent");
    REQUIRE(a->t < a->T, B200RL_ERR_INVALID, "rollout is full");
    a->t += 1;
    b200rl_env_internal_set_traj_targets(a->env, nullptr, nullptr);
    return B200RL_OK;
}
/* n x (plan! -> act! -> push!) without leaving the device */
int b200rl_onpolicy_collect(b200rl_onpolicy* a, int n_steps) {
    REQUIRE(a && n_steps >= 0, B200RL_ERR_INVALID, "bad argument");
    if (n_steps > 0 && nn_tc_enabled() && fused_rollout_enabled()) {   // one launch for the whole stretch (fwd_tc.cu)
        REQUIRE(a->t + n_steps <= a->T, B200RL_ERR_INVALID, "rollout is full: call b200rl_onpolicy_update first");
        TRY(ctx_bind(a->ctx));
        const AcHyper hp = hyper_of(a->cfg);
        const int fin = a->t + n_steps == a->T ? 1 : 0;
        int st = nn_tc_rollout(a->ctx, a->env, a->net->actor, a->net->critic, a->net->params, hp, a->rng, a->t, n_steps, a->T, fin, a->states,
                               a->actions, a->logp, a->values, a->rewards, a->terminals);
        if (st == B200RL_OK) {
            a->t += n_steps;
            a->bootstrap_done = fin != 0;
            return B200RL_OK;
        }
        if (st != B200RL_ERR_UNSUPPORTED) return st;
    }
    for (int k = 0; k < n_steps; ++k) {
        TRY(b200rl_onpolicy_plan(a, nullptr));
        TRY(b200rl_onpolicy_act(a));
        TRY(b200rl_onpolicy_push(a));
    }
    return B200RL_OK;
}
int b200rl_onpolicy_fill(b200rl_onpolicy* a, int* t_out, int* T_out) {
    REQUIRE(a, B200RL_ERR_INVALID, "null agent");
    if (t_out) *t_out = a->t;
    if (T_out) *T_out = a->T;
    return B200RL_OK;
}

/* optimise!(agent): V(s_{T+1}), GAE (+returns, advantage normalisation), then n_epochs x
 * n_microbatches of {loss+grad, reduce, [all-reduce], clip + Adam}.  perm_host: optional
 * (n_epochs, N*T) int32 0-based permutations (the host's shuffle!); NULL = device Feistel
 * permutation keyed by (update counter, epoch).  stats_host: optional (n_epochs*n_microbatches, 6)
 * floats [actor_loss, critic_loss, entropy, loss, grad_norm, 0] (forces a sync). */
int b200rl_onpolicy_update(b200rl_onpolicy* a, const int32_t* perm_host, float* stats_host) {
    REQUIRE(a, B200RL_ERR_INVALID, "null agent");
    REQUIRE(a->t == a->T, B200RL_ERR_INVALID, "rollout not full yet");
    TRY(ctx_bind(a->ctx));
    b200rl_ctx* ctx = a->ctx;
    b200rl_net* n = a->net;
    const b200rl_onpolicy_config& c = a->cfg;
    int64_t N = a->N, T = a->T, NT_ = N * T;
    int world = b200rl_comm_world(ctx);
    // measurement aid (b200rl_debug_phase_slots): events between the phases, eager path only
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    CUDA_TRY(cudaStreamIsCapturing(ctx->stream, &cap));
    const int pb = (cap == cudaStreamCaptureStatusNone && ctx->phase_base + 3 + 2 * a->stats_rows <= b200rl_ctx::kTimerSlots) ? ctx->phase_base : -1;
    auto phase = [&](int k) -> int { return pb >= 0 ? b200rl_timer_record(ctx, pb + k) : B200RL_OK; };
    TRY(phase(0));
    // bootstrap value of the state after the last step
    const float* obs = (const float*)env_field(a->env, B200RL_FIELD_OBS);
    // (a copy kernel, not cudaMemcpyAsync D2D: device-to-device copies are on CUDA's implicit-synchronisation list)
    if (!a->bootstrap_done) {   // (the fused rollout has already written column T of states / values)
        copy_f32_kernel<<<grid_for(N * a->ns, 256), 256, 0, ctx->stream>>>(a->states + (size_t)N * a->ns * T, obs, N * a->ns);
        LAUNCH_CHECK(ctx);
        TRY(nn_mlp_forward(ctx, n->critic, n->params + n->actor.nparams(), obs, N, a->values + (size_t)N * T));
    }
    a->bootstrap_done = false;
    // GAE + returns + normalisation sums
    int n_part = b200rl_gae_fused_partials_count(N) / 2;
    TRY(b200rl_gae_fused_internal(ctx, a->adv, a->ret, a->rewards, a->values, a->terminals, c.gamma, c.lambda, N, T,
                                  c.normalize_advantage ? a->norm_partials : nullptr, nullptr));
    if (c.algo == 1) {  // A2C: critic target = discounted gains bootstrapped with V(s_{T+1})
        TRY(b200rl_discount_rewards_f32(ctx, a->ret, a->rewards, a->terminals, a->values + (size_t)N * T, c.gamma, N, T, 2, 1));
    }
    if (c.normalize_advantage) {
        sum_norm_partials_kernel<<<1, 32, 0, ctx->stream>>>(a->norm_partials, n_part, a->norm_sums);
        LAUNCH_CHECK(ctx);
        if (world > 1) TRY(b200rl_comm_allreduce_internal(ctx, a->norm_sums, 2, 1));
        finalize_norm2_kernel<<<1, 32, 0, ctx->stream>>>(a->norm_sums, (double)NT_ * (double)world, a->norm2);
        LAUNCH_CHECK(ctx);
    }
    {   // one 32-byte record per sample for the permuted minibatch gathers (n_epochs x n_microbatches of them follow)
        const unsigned g = grid_for(NT_, 256);
        const uint32_t* act = (const uint32_t*)a->actions;
        switch (a->ns) {
            case 1: pack_records_kernel<1><<<g, 256, 0, ctx->stream>>>(a->rec, a->states, act, a->logp, a->adv, a->ret, NT_); break;
            case 2: pack_records_kernel<2><<<g, 256, 0, ctx->stream>>>(a->rec, a->states, act, a->logp, a->adv, a->ret, NT_); break;
            case 3: pack_records_kernel<3><<<g, 256, 0, ctx->stream>>>(a->rec, a->states, act, a->logp, a->adv, a->ret, NT_); break;
            default: pack_records_kernel<4><<<g, 256, 0, ctx->stream>>>(a->rec, a->states, act, a->logp, a->adv, a->ret, NT_); break;
        }
        LAUNCH_CHECK(ctx);
    }
    if (perm_host) {
        CUDA_TRY(cudaMemcpyAsync(a->perm_dev, perm_host, (size_t)c.n_epochs * NT_ * 4, cudaMemcpyHostToDevice, ctx->stream));
    }
    TRY(phase(1));
    const AcHyper hp = hyper_of(c);
    const int64_t B = minibatch_size(a);
    const OptPath path = onpolicy_opt_path(a);
    int row = 0;
    for (int e = 0; e < c.n_epochs; ++e) {
        for (int mb = 0; mb < c.n_microbatches; ++mb, ++row) {
            // permutation key = n_updates * 1000003 + e * 7919 + 12345; the update counter is read from device memory (upd_dev)
            // so that a captured iteration can be replayed
            AcBatch b{a->states, a->ns, a->actions, a->logp, a->adv, a->ret,
                      perm_host ? a->perm_dev + (size_t)e * NT_ + (size_t)mb * B : nullptr,
                      (uint32_t)NT_, (uint32_t)e * 7919u + 12345u, (uint32_t)(mb * B), a->upd_dev, a->rec, B,
                      1.0f / ((float)B * (float)world), a->norm2};
            float* stats_row = a->stats_dev + (size_t)row * 8;
            unsigned int* tick = row == a->stats_rows - 1 ? a->upd_dev : nullptr;   // the last optimiser step closes the update
            const OptStep st = net_opt_state(n, c, c.lr, stats_row, tick);
            if (path == OPT_FUSED_TAIL) {   // one launch: loss + backward + [peer exchange] + clip + Adam
                const int ctas = nn_ac_loss_grad_step(ctx, n->actor, n->critic, hp, b, n->partial, n->loss_partial, st);
                if (ctas < 0) return ctas;
                TRY(phase(2 + 2 * row));
            } else {
                const int ctas = nn_ac_loss_grad(ctx, n->actor, n->critic, n->params, hp, b, n->partial, n->loss_partial);
                if (ctas < 0) return ctas;
                TRY(phase(2 + 2 * row));
                TRY(net_opt_step(n, path, ctas, 2 * ctas, st));
            }
            TRY(phase(3 + 2 * row));
            n->n_updates += 1;
        }
    }
    a->n_updates += 1;
    a->t = 0;
    if (stats_host) TRY(onpolicy_read_stats(a, stats_host));
    return B200RL_OK;
}

/* n_iters x { collect(T); update } — the whole PPO / A2C iteration (fused rollout, bootstrap, GAE, record packing, n_epochs x
 * n_microbatches x {loss + backward, [peer exchange +] clip + Adam}) replayed as ONE CUDA graph launch per iteration, so
 * the ranks of a sharded run cannot drift apart on host launch jitter (they meet 17 times per iteration inside the peer
 * exchange).  Needs an empty rollout (t = 0).  Every per-launch counter lives in device memory (update counter, exchange
 * sequence numbers, self-resetting grid barrier), so the captured launches are replayable as they are.  The first
 * iteration ever runs eagerly (lazy module loading, scratch growth, function attributes), the second is captured.
 * stats_host: optional (n_epochs * n_microbatches, 6) rows of the LAST iteration (forces a sync).
 * Falls back to eager launches when capture is impossible (NCCL path without the peer exchange, B200RL_GRAPH=0). */
int b200rl_onpolicy_iterate(b200rl_onpolicy* a, int n_iters, float* stats_host) {
    REQUIRE(a && n_iters >= 0, B200RL_ERR_INVALID, "bad argument");
    REQUIRE(a->t == 0, B200RL_ERR_INVALID, "iterate needs an empty rollout (t = 0)");
    TRY(ctx_bind(a->ctx));
    b200rl_ctx* ctx = a->ctx;
    static int graph_env = -1;
    if (graph_env < 0) { const char* e = getenv("B200RL_GRAPH"); graph_env = (e && e[0] == '0') ? 0 : 1; }
    const bool capturable = graph_env && !a->graph_failed && ctx->phase_base < 0 && onpolicy_opt_path(a) != OPT_NCCL_CHAIN;
    const int rows = a->stats_rows;
    for (int it = 0; it < n_iters; ++it) {
        if (!capturable || !a->warmed) {
            TRY(b200rl_onpolicy_collect(a, a->T));
            TRY(b200rl_onpolicy_update(a, nullptr, nullptr));
            a->warmed = true;
            continue;
        }
        const int tc_now = nn_tc_enabled() ? 1 : 0;
        const uint64_t env_gen = (uint64_t)b200rl_env_internal_max_timeout(a->env);
        if (a->graph_exec && (a->graph_tc != tc_now || a->graph_env_gen != env_gen)) {   // a launch argument changed: re-capture
            cudaGraphExecDestroy(a->graph_exec); a->graph_exec = nullptr;
            cudaGraphDestroy(a->graph); a->graph = nullptr;
        }
        if (!a->graph_exec) {
            // capture does not execute: the host-side bookkeeping the captured calls did is rolled back and redone per replay
            const uint64_t l0 = ctx->launches, nu0 = a->n_updates, nnu0 = a->net->n_updates;
            CUDA_TRY(cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal));
            int st = b200rl_onpolicy_collect(a, a->T);
            if (st == B200RL_OK) st = b200rl_onpolicy_update(a, nullptr, nullptr);
            cudaGraph_t g = nullptr;
            cudaError_t ce = cudaStreamEndCapture(ctx->stream, &g);
            a->graph_launches = ctx->launches - l0;
            ctx->launches = l0; a->n_updates = nu0; a->net->n_updates = nnu0; a->t = 0; a->bootstrap_done = false;
            b200rl_env_internal_add_steps(a->env, (uint64_t)0 - (uint64_t)a->T);
            if (st != B200RL_OK || ce != cudaSuccess || !g) {
                if (g) cudaGraphDestroy(g);
                cudaGetLastError();
                a->graph_failed = 1;   // stay on eager launches
                TRY(b200rl_onpolicy_collect(a, a->T));
                TRY(b200rl_onpolicy_update(a, nullptr, nullptr));
                continue;
            }
            cudaError_t ie = cudaGraphInstantiate(&a->graph_exec, g, 0);
            if (ie != cudaSuccess) {
                cudaGraphDestroy(g);
                cudaGetLastError();
                a->graph_exec = nullptr; a->graph_failed = 1;
                TRY(b200rl_onpolicy_collect(a, a->T));
                TRY(b200rl_onpolicy_update(a, nullptr, nullptr));
                continue;
            }
            a->graph = g; a->graph_tc = tc_now; a->graph_env_gen = env_gen;
        }
        CUDA_TRY(cudaGraphLaunch(a->graph_exec, ctx->stream));
        ctx->launches += a->graph_launches;
        a->n_updates += 1; a->net->n_updates += (uint64_t)rows;
        b200rl_env_internal_add_steps(a->env, (uint64_t)a->T);
    }
    if (stats_host && n_iters > 0) TRY(onpolicy_read_stats(a, stats_host));
    return B200RL_OK;
}
/* 1 when b200rl_onpolicy_iterate replays a captured graph, 0 when it launches eagerly (diagnostic for tests / bench) */
int b200rl_onpolicy_graph_active(b200rl_onpolicy* a, int* out) {
    REQUIRE(a && out, B200RL_ERR_INVALID, "null argument");
    *out = a->graph_exec ? 1 : 0;
    return B200RL_OK;
}

/* rollout tensors for inspection / parity tests.  field: 0 state (ns, N, T+1) | 1 action (N, T) |
 * 2 logp (N, T) | 3 reward (N, T) | 4 terminal (N, T) u8 | 5 value (N, T+1) | 6 advantage (N, T) |
 * 7 return (N, T) | 8 policy rng (4, N) u64 | 9 advantage norm {mean, inv_std} */
int b200rl_onpolicy_get(b200rl_onpolicy* a, int field, void* host_dst, size_t bytes) {
    REQUIRE(a && host_dst, B200RL_ERR_INVALID, "null argument");
    TRY(ctx_bind(a->ctx));
    size_t N = (size_t)a->N, T = (size_t)a->T;
    const void* src = nullptr;
    size_t need = 0;
    switch (field) {
        case 0: src = a->states; need = N * a->ns * (T + 1) * 4; break;
        case 1: src = a->actions; need = N * T * 4; break;
        case 2: src = a->logp; need = N * T * 4; break;
        case 3: src = a->rewards; need = N * T * 4; break;
        case 4: src = a->terminals; need = N * T; break;
        case 5: src = a->values; need = N * (T + 1) * 4; break;
        case 6: src = a->adv; need = N * T * 4; break;
        case 7: src = a->ret; need = N * T * 4; break;
        case 8: src = a->rng; need = N * 32; break;
        case 9: src = a->norm2; need = 8; break;
        default: REQUIRE(false, B200RL_ERR_INVALID, "unknown field");
    }
    REQUIRE(bytes >= need, B200RL_ERR_INVALID, "destination too small");
    CUDA_TRY(cudaMemcpyAsync(host_dst, src, need, cudaMemcpyDeviceToHost, a->ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(a->ctx->stream));
    return B200RL_OK;
}

/* checkpoint import: fields 0-5 and 8 of b200rl_onpolicy_get (advantages / returns / normalisation are recomputed by update) */
int b200rl_onpolicy_set(b200rl_onpolicy* a, int field, const void* host_src, size_t bytes) {
    REQUIRE(a && host_src, B200RL_ERR_INVALID, "null argument");
    TRY(ctx_bind(a->ctx));
    size_t N = (size_t)a->N, T = (size_t)a->T;
    void* dst = nullptr;
    size_t need = 0;
    switch (field) {
        case 0: dst = a->states; need = N * a->ns * (T + 1) * 4; break;
        case 1: dst = a->actions; need = N * T * 4; break;
        case 2: dst = a->logp; need = N * T * 4; break;
        case 3: dst = a->rewards; need = N * T * 4; break;
        case 4: dst = a->terminals; need = N * T; break;
        case 5: dst = a->values; need = N * (T + 1) * 4; break;
        case 8: dst = a->rng; need = N * 32; break;
        default: REQUIRE(false, B200RL_ERR_INVALID, "field not settable");
    }
    REQUIRE(bytes >= need, B200RL_ERR_INVALID, "source too small");
    CUDA_TRY(cudaMemcpyAsync(dst, host_src, need, cudaMemcpyHostToDevice, a->ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(a->ctx->stream));
    return B200RL_OK;
}
int b200rl_onpolicy_export_state(b200rl_onpolicy* a, int64_t* c3) {
    REQUIRE(a && c3, B200RL_ERR_INVALID, "null argument");
    c3[0] = a->t; c3[1] = (int64_t)a->n_updates; c3[2] = (int64_t)a->net->n_updates;
    return B200RL_OK;
}
int b200rl_onpolicy_import_state(b200rl_onpolicy* a, const int64_t* c3) {
    REQUIRE(a && c3, B200RL_ERR_INVALID, "null argument");
    REQUIRE(c3[0] >= 0 && c3[0] <= a->T && c3[1] >= 0 && c3[2] >= 0, B200RL_ERR_INVALID, "counters out of range");
    a->t = (int)c3[0]; a->n_updates = (uint64_t)c3[1]; a->net->n_updates = (uint64_t)c3[2];
    TRY(ctx_bind(a->ctx));
    const unsigned int upd = (unsigned int)a->n_updates;   // the device copy keys the minibatch permutation
    CUDA_TRY(cudaMemcpyAsync(a->upd_dev, &upd, sizeof upd, cudaMemcpyHostToDevice, a->ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(a->ctx->stream));
    a->bootstrap_done = false;   // column T of states / values is rewritten from the env's observation by the next update
    b200rl_env_internal_set_traj_targets(a->env, nullptr, nullptr);
    return B200RL_OK;
}

/* Measurement aid (bench.py roofline): average device time of `reps` back-to-back launches of one
 * hot-path kernel on the agent's current tensors, CUDA events on the ctx stream.
 * which: 0 loss+backward minibatch kernel (K7) | 1 policy inference (K6) | 2 env step (K1, mutates the env) |
 * 3 fused GAE (K5) | 4 partial reduce + clip + Adam (K8) */
int b200rl_onpolicy_time_kernel(b200rl_onpolicy* a, int which, int reps, float* avg_ms_out) {
    REQUIRE(a && avg_ms_out && reps >= 1, B200RL_ERR_INVALID, "bad argument");
    TRY(ctx_bind(a->ctx));
    b200rl_ctx* ctx = a->ctx;
    b200rl_net* n = a->net;
    const b200rl_onpolicy_config& c = a->cfg;
    int64_t N = a->N, T = a->T, NT_ = N * T, B = NT_ / c.n_microbatches;
    const AcHyper hp = hyper_of(c);
    const float* obs = (const float*)env_field(a->env, B200RL_FIELD_OBS);
    const int ctas = nn_ac_partial_rows(ctx, n->actor, n->critic, hp, B);
    void* rng_copy = nullptr;
    if (which == 1) {
        TRY(ctx_scratch(ctx, (size_t)N * 32 + (size_t)N * 12 + 256, &rng_copy));
        CUDA_TRY(cudaMemcpyAsync(rng_copy, a->rng, (size_t)N * 32, cudaMemcpyDeviceToDevice, ctx->stream));
    }
    auto once = [&]() -> int {
        switch (which) {
            case 0: {
                AcBatch b{a->states, a->ns, a->actions, a->logp, a->adv, a->ret, nullptr, (uint32_t)NT_, 12345u, 0u, nullptr, a->rec, B, 1.0f / (float)B,
                          a->norm2};
                int st = nn_ac_loss_grad(ctx, n->actor, n->critic, n->params, hp, b, n->partial, n->loss_partial);
                return st < 0 ? st : B200RL_OK;
            }
            case 1: {
                float* o = (float*)((char*)rng_copy + (size_t)N * 32);
                return nn_policy_act(ctx, n->actor, n->critic, n->params, hp, obs, N, (unsigned long long*)rng_copy, o, o + N, o + 2 * N, nullptr, nullptr);
            }
            case 2: return b200rl_env_step(a->env, a->actions, 1, 1);
            case 3: return b200rl_gae_fused_internal(ctx, a->adv, a->ret, a->rewards, a->values, a->terminals, c.gamma, c.lambda, N, T, a->norm_partials, nullptr);
            case 4:   // the unfused optimiser step as update() runs it (lr = 0: parameters stay put), incl. the exchange of a sharded run
                return net_opt_step(n, net_opt_path(n, false, hp, B), ctas, 2 * ctas, net_opt_state(n, c, 0.0f, nullptr, nullptr));
        }
        b200rl_set_error("unknown kernel id");
        return B200RL_ERR_INVALID;
    };
    REQUIRE(!(which == 2 && a->continuous), B200RL_ERR_UNSUPPORTED, "env-step timing uses the discrete action column");
    TRY(once());  // warm-up
    CUDA_TRY(cudaEventRecord(ctx->ev0, ctx->stream));
    for (int r = 0; r < reps; ++r) TRY(once());
    CUDA_TRY(cudaEventRecord(ctx->ev1, ctx->stream));
    CUDA_TRY(cudaEventSynchronize(ctx->ev1));
    float ms = 0.f;
    CUDA_TRY(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    *avg_ms_out = ms / (float)reps;
    return B200RL_OK;
}

// ------------------------------------------------------------------ DQN ---------------------
/* push!(trajectory, env): append the env's last transition (action, reward, terminal, next obs) — all on device.
 * first_state_only 1: episode-start frame for every lane (PreEpisodeStage); 2: only for the lanes whose last transition was terminal */
int b200rl_traj_push_env(b200rl_traj* t, b200rl_env* env, int first_state_only) {
    REQUIRE(t && env, B200RL_ERR_INVALID, "null argument");
    REQUIRE(b200rl_traj_internal_lanes(t) == b200rl_env_internal_n(env), B200RL_ERR_INVALID, "trajectory lanes != number of envs");
    REQUIRE(b200rl_env_internal_dtype(env) == B200RL_F32, B200RL_ERR_UNSUPPORTED, "the trajectory stores Float32 states: construct the env with T = Float32");
    const float* obs = (const float*)env_field(env, B200RL_FIELD_OBS);
    if (first_state_only == 2) return b200rl_traj_push_episode_start(t, obs, 1, 1);   // only the lanes whose episode has ended (soft reset)
    if (first_state_only) return b200rl_traj_push_state(t, obs, 1);
    return b200rl_traj_push(t, (const int32_t*)env_field(env, B200RL_FIELD_ACTION), (const float*)env_field(env, B200RL_FIELD_REWARD),
                            (const uint8_t*)env_field(env, B200RL_FIELD_FLAGS), obs, 1);
}

/* optimise!(DQNLearner / PrioritizedDQNLearner, batch): sample + gather (K4), TD loss + backward
 * (K7), clip + Adam (K8), priority write-back, target sync every target_update_freq updates.
 * stats_host[4] = loss, grad_norm, mean |td|, n_updates (NULL = no sync). */
int b200rl_dqn_update(b200rl_net* n, b200rl_traj* t, const b200rl_dqn_config* cfg, float* stats_host) {
    REQUIRE(n && t && cfg && n->kind == 2, B200RL_ERR_INVALID, "bad argument (needs a Q-network)");
    REQUIRE(n->ctx == b200rl_traj_internal_ctx(t), B200RL_ERR_INVALID, "net/trajectory belong to different ctx");
    TRY(ctx_bind(n->ctx));
    b200rl_ctx* ctx = n->ctx;
    TRY(b200rl_traj_sample(t, cfg->per_beta));
    TrajBatchView b = b200rl_traj_internal_batch(t);
    REQUIRE(b.ns == n->actor.in, B200RL_ERR_INVALID, "state width mismatch");
    void* sc;
    // scratch: [Q tables: 2*B*nout] used inside nn_dqn_loss_grad, td after them
    size_t q_bytes = (size_t)b.B * n->actor.nout * 4 * 2 + 256;
    TRY(ctx_scratch(ctx, q_bytes + (size_t)b.B * 4 + 256, &sc));
    float* td = (float*)((char*)sc + q_bytes);
    int world = b200rl_comm_world(ctx);
    int np_ = nn_dqn_loss_grad(ctx, n->actor, n->params, n->target, b.s, b.a, b.r, b.t, b.s2, b.w, b.B, 1.0f / ((float)b.B * (float)world), cfg->gamma,
                               cfg->huber, cfg->double_dqn, n->partial, n->loss_partial, td);
    if (np_ < 0) return np_;
    TRY(net_opt_step(n, net_opt_path(n, false, AcHyper{}, b.B), np_, np_, net_opt_state(n, *cfg, cfg->lr, nullptr, nullptr)));
    if (b200rl_traj_internal_prioritized(t)) TRY(b200rl_traj_internal_priority_from_td(t, td, cfg->per_eps, cfg->per_alpha));
    n->n_updates += 1;
    if (cfg->target_update_freq > 0 && n->n_updates % (uint64_t)cfg->target_update_freq == 0) TRY(nn_target_sync(ctx, n->target, n->params, n->np, cfg->rho));
    if (stats_host) {
        float l4[4], gn;
        std::vector<float> tdh((size_t)b.B);
        CUDA_TRY(cudaMemcpyAsync(l4, n->loss4, 16, cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(cudaMemcpyAsync(&gn, n->gnorm, 4, cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(cudaMemcpyAsync(tdh.data(), td, (size_t)b.B * 4, cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(cudaStreamSynchronize(ctx->stream));
        double s = 0;
        for (float x : tdh) s += x < 0 ? -x : x;
        stats_host[0] = l4[0] / ((float)b.B * (float)world); stats_host[1] = gn; stats_host[2] = (float)(s / (double)b.B);
        stats_host[3] = (float)n->n_updates;
    }
    return B200RL_OK;
}
/* TD errors (B floats) of the batch used by the last b200rl_dqn_update (for parity tests) */
int b200rl_dqn_last_td(b200rl_net* n, b200rl_traj* t, float* host_dst, int64_t count) {
    REQUIRE(n && t && host_dst, B200RL_ERR_INVALID, "null argument");
    TRY(ctx_bind(n->ctx));
    TrajBatchView b = b200rl_traj_internal_batch(t);
    REQUIRE(count >= b.B, B200RL_ERR_INVALID, "destination too small");
    size_t q_bytes = (size_t)b.B * n->actor.nout * 4 * 2 + 256;
    REQUIRE(n->ctx->scratch_bytes >= q_bytes + (size_t)b.B * 4, B200RL_ERR_INVALID, "no update has run yet");
    CUDA_TRY(cudaMemcpyAsync(host_dst, (char*)n->ctx->scratch + q_bytes, (size_t)b.B * 4, cudaMemcpyDeviceToHost, n->ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(n->ctx->stream));
    return B200RL_OK;
}

}  // extern "C"
