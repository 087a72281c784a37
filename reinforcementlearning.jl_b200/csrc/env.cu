// env.cu — K1/K2: batched classic-control env step, reset and fused random policy.
//
// One thread per env, 256 threads per CTA.  State is (NS, N) column-major so one env's state
// is one 16-byte (Float32 CartPole: float4) or 8-byte vector; reward/flags/t are SoA vectors;
// the per-env Xoshiro256++ state is 32 B AoS and is only touched by threads that draw.
// Arithmetic follows the reference line by line with Julia's promotion rules (which
// sub-expressions are Float64 for T = Float32) — see DESIGN.md §K1 and
//   RLEnvs/src/environments/examples/CartPoleEnv.jl:98-140
//   RLEnvs/src/environments/examples/PendulumEnv.jl:84-122
//   RLEnvs/src/environments/examples/MountainCarEnv.jl:99-135
// Compiled with -fmad=false (no contraction; Julia never contracts) and IEEE div.
#include <type_traits>

#include "common.cuh"
#include "env_device.cuh"
#include "internal.h"

using jld::Xo;
using namespace envdev;

namespace {

constexpr int kBlock = 256;

// ------------------------------------------------------------------ kernels -----------
// Block-level accumulation of episode statistics: one atomicAdd triple per CTA that saw a
// finished episode (device-side TotalRewardPerEpisode / BatchStepsPerEpisode, hooks.jl:146-231).
__device__ __forceinline__ void block_episode_stats(double* stats, bool finished, float ret, int len) {
    __shared__ float s_ret[kBlock / 32];
    __shared__ int s_len[kBlock / 32];
    __shared__ int s_cnt[kBlock / 32];
    unsigned m = __ballot_sync(0xffffffffu, finished);
    float r = finished ? ret : 0.f;
    int l = finished ? len : 0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        r += __shfl_xor_sync(0xffffffffu, r, o);
        l += __shfl_xor_sync(0xffffffffu, l, o);
    }
    int w = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) { s_ret[w] = r; s_len[w] = l; s_cnt[w] = __popc(m); }
    __syncthreads();
    if (threadIdx.x == 0) {
        double rr = 0; long long ll = 0; int cc = 0;
#pragma unroll
        for (int k = 0; k < kBlock / 32; ++k) { rr += s_ret[k]; ll += s_len[k]; cc += s_cnt[k]; }
        if (cc) {
            atomicAdd(&stats[0], (double)cc);
            atomicAdd(&stats[1], rr);
            atomicAdd(&stats[2], (double)ll);
        }
    }
}

template <class Env, bool RANDOM, bool AUTO>
__global__ void __launch_bounds__(kBlock) env_step_kernel(typename Env::P p, EnvArrays a, int64_t N, const void* actions_v) {
    using T = typename Env::real;
    using act_t = typename Env::act_t;
    int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    bool active = i < N;
    bool finished = false;
    float fin_ret = 0.f;
    int fin_len = 0;
    if (active) {
        typename Env::S s = Env::load(a.state, i);
        int t = a.t[i];
        uint8_t prev = a.flags[i];
        Xo g;
        bool have_rng = false;
        act_t act;
        bool ok = true;
        if (RANDOM) {  // plan!(RandomPolicy): rand(rng, Base.OneTo(n)) on the env's own stream
            g = load_rng(a.rng, i);
            have_rng = true;
            act = Env::from_index(p, jld::rand_oneto(g, Env::n_random(p)));
        } else {
            act = reinterpret_cast<const act_t*>(actions_v)[i];
            ok = Env::valid(p, act);
            if (!ok) *a.err = 1;  // `@assert a in action_space(env)` -> flag, env left untouched
        }
        if (ok) {
            bool done;
            T rew;
            Env::step(p, s, t, act, done, rew);
            // MaxTimeoutEnv: terminated also when current_t (= t + 1) > max_t; reward untouched
            if (a.max_timeout > 0 && t + 1 > a.max_timeout) done = true;
            float ret = a.ep_ret[i] + (float)rew;
            uint8_t f = done ? 1 : 0;
            if (done && !((prev & 1) && !(prev & 2))) { finished = true; fin_ret = ret; fin_len = t; }
            if (done) ret = 0.f;
            if (AUTO && done) {  // fused soft reset (MultiThreadEnv reset!(env; is_force=false))
                if (!have_rng) { g = load_rng(a.rng, i); have_rng = true; }
                Env::reset(p, s, g, act);
                t = 0;
                f = 3;
            }
            Env::store(a.state, i, s);
            if (!Env::kObsIsState) Env::write_obs(a.obs, i, N, s);
            a.t[i] = t;
            a.flags[i] = f;
            reinterpret_cast<T*>(a.reward)[i] = rew;
            reinterpret_cast<act_t*>(a.action)[i] = act;
            a.ep_ret[i] = ret;
            if (a.traj_reward) reinterpret_cast<T*>(a.traj_reward)[i] = rew;
            if (a.traj_terminal) a.traj_terminal[i] = done ? 1 : 0;
        }
        if (have_rng) store_rng(a.rng, i, g);
    }
    block_episode_stats(a.stats, finished, fin_ret, fin_len);
}

// envs whose reset! also sets the reward field (AcrobotEnv.jl:105: env.reward = -1); the others derive reward(env) from `done`
template <class Env> struct ResetReward { static constexpr bool set = false; static __device__ double value() { return 0.0; } };
template <> struct ResetReward<AcrobotD> { static constexpr bool set = true; static __device__ double value() { return -1.0; } };

template <class Env>
__global__ void __launch_bounds__(kBlock) env_reset_kernel(typename Env::P p, EnvArrays a, int64_t N, int force) {
    using act_t = typename Env::act_t;
    int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (i >= N) return;
    uint8_t f = a.flags[i];
    if (force || ((f & 1) && !(f & 2))) {
        typename Env::S s = Env::load(a.state, i);
        Xo g = load_rng(a.rng, i);
        act_t act = reinterpret_cast<act_t*>(a.action)[i];
        Env::reset(p, s, g, act);
        store_rng(a.rng, i, g);
        Env::store(a.state, i, s);
        if (!Env::kObsIsState) Env::write_obs(a.obs, i, N, s);
        a.t[i] = 0;
        reinterpret_cast<act_t*>(a.action)[i] = act;
        a.ep_ret[i] = 0.f;
        if (ResetReward<Env>::set) reinterpret_cast<typename Env::real*>(a.reward)[i] = (typename Env::real)ResetReward<Env>::value();
    }
    a.flags[i] = 0;
}

}  // namespace

// ------------------------------------------------------------------ handle ------------
struct b200rl_env {
    b200rl_ctx* ctx;
    int kind, dtype;
    int64_t N;
    int ns, nobs;
    bool continuous;
    size_t tsize;
    union {
        CartPoleD<float>::P cp32;
        CartPoleD<double>::P cp64;
        PendP pend;
        MountainCarD<false>::P mc;
        PendPT<double> pend64;
        MountainCarPT<double> mc64;
        AcrobotP acro;
    } p;
    size_t asize;   // bytes per stored action (8 for a Float64 continuous action space, else 4)
    EnvArrays a;
    uint64_t steps_launched;
};

template <class Env> static int launch_step(b200rl_env* e, const typename Env::P& p, const void* actions, bool random, bool auto_reset) {
    unsigned grid = grid_for(e->N, kBlock);
    cudaStream_t st = e->ctx->stream;
    if (random) {
        if (auto_reset) env_step_kernel<Env, true, true><<<grid, kBlock, 0, st>>>(p, e->a, e->N, nullptr);
        else env_step_kernel<Env, true, false><<<grid, kBlock, 0, st>>>(p, e->a, e->N, nullptr);
    } else {
        if (auto_reset) env_step_kernel<Env, false, true><<<grid, kBlock, 0, st>>>(p, e->a, e->N, actions);
        else env_step_kernel<Env, false, false><<<grid, kBlock, 0, st>>>(p, e->a, e->N, actions);
    }
    LAUNCH_CHECK(e->ctx);
    return B200RL_OK;
}
template <class Env> static int launch_reset(b200rl_env* e, const typename Env::P& p, int force) {
    env_reset_kernel<Env><<<grid_for(e->N, kBlock), kBlock, 0, e->ctx->stream>>>(p, e->a, e->N, force);
    LAUNCH_CHECK(e->ctx);
    return B200RL_OK;
}

static int dispatch_step(b200rl_env* e, const void* actions, bool random, bool auto_reset) {
    switch (e->kind) {
        case B200RL_ENV_CARTPOLE:
            if (e->dtype == B200RL_F64) return launch_step<CartPoleD<double>>(e, e->p.cp64, actions, random, auto_reset);
            if (e->continuous && !random) {
                CartPoleD<float, true>::P q;
                static_assert(sizeof(q) == sizeof(e->p.cp32), "same params layout");
                memcpy(&q, &e->p.cp32, sizeof q);
                return launch_step<CartPoleD<float, true>>(e, q, actions, random, auto_reset);
            }
            return launch_step<CartPoleD<float>>(e, e->p.cp32, actions, random, auto_reset);
        case B200RL_ENV_PENDULUM:
            if (e->dtype == B200RL_F64) {
                if (e->continuous && !random) return launch_step<PendulumD<true, double>>(e, e->p.pend64, actions, random, auto_reset);
                return launch_step<PendulumD<false, double>>(e, e->p.pend64, actions, random, auto_reset);
            }
            if (e->continuous && !random) return launch_step<PendulumD<true>>(e, e->p.pend, actions, random, auto_reset);
            return launch_step<PendulumD<false>>(e, e->p.pend, actions, random, auto_reset);
        case B200RL_ENV_MOUNTAINCAR:
            if (e->dtype == B200RL_F64) {
                if (e->continuous && !random) return launch_step<MountainCarD<true, double>>(e, e->p.mc64, actions, random, auto_reset);
                return launch_step<MountainCarD<false, double>>(e, e->p.mc64, actions, random, auto_reset);
            }
            if (e->continuous && !random) {
                MountainCarD<true>::P q;
                static_assert(sizeof(q) == sizeof(e->p.mc), "same params layout");
                memcpy(&q, &e->p.mc, sizeof q);
                return launch_step<MountainCarD<true>>(e, q, actions, random, auto_reset);
            }
            return launch_step<MountainCarD<false>>(e, e->p.mc, actions, random, auto_reset);
        case B200RL_ENV_ACROBOT:
            return launch_step<AcrobotD>(e, e->p.acro, actions, random, auto_reset);
    }
    return B200RL_ERR_INVALID;
}
static int dispatch_reset(b200rl_env* e, int force) {
    switch (e->kind) {
        case B200RL_ENV_CARTPOLE:
            if (e->dtype == B200RL_F64) return launch_reset<CartPoleD<double>>(e, e->p.cp64, force);
            if (e->continuous) {
                CartPoleD<float, true>::P q;
                memcpy(&q, &e->p.cp32, sizeof q);
                return launch_reset<CartPoleD<float, true>>(e, q, force);
            }
            return launch_reset<CartPoleD<float>>(e, e->p.cp32, force);
        case B200RL_ENV_PENDULUM:
            if (e->dtype == B200RL_F64)
                return e->continuous ? launch_reset<PendulumD<true, double>>(e, e->p.pend64, force) : launch_reset<PendulumD<false, double>>(e, e->p.pend64, force);
            return launch_reset<PendulumD<true>>(e, e->p.pend, force);
        case B200RL_ENV_MOUNTAINCAR:
            if (e->dtype == B200RL_F64)
                return e->continuous ? launch_reset<MountainCarD<true, double>>(e, e->p.mc64, force) : launch_reset<MountainCarD<false, double>>(e, e->p.mc64, force);
            return launch_reset<MountainCarD<false>>(e, e->p.mc, force);
        case B200RL_ENV_ACROBOT:
            return launch_reset<AcrobotD>(e, e->p.acro, force);
    }
    return B200RL_ERR_INVALID;
}

static size_t field_bytes(const b200rl_env* e, int field) {
    size_t N = (size_t)e->N;
    switch (field) {
        case B200RL_FIELD_STATE: return N * e->ns * e->tsize;
        case B200RL_FIELD_OBS: return N * e->nobs * e->tsize;
        case B200RL_FIELD_REWARD: return N * e->tsize;
        case B200RL_FIELD_TERMINAL: case B200RL_FIELD_FLAGS: return N;
        case B200RL_FIELD_T: return N * 4;
        case B200RL_FIELD_RNG: return N * 32;
        case B200RL_FIELD_ACTION: return N * e->asize;
        case B200RL_FIELD_EPISODE_RETURN: return N * 4;
        case B200RL_FIELD_EPISODE_STATS: return 4 * sizeof(double);
    }
    return 0;
}
static void* field_ptr(const b200rl_env* e, int field) {
    switch (field) {
        case B200RL_FIELD_STATE: return e->a.state;
        case B200RL_FIELD_OBS: return e->a.obs;
        case B200RL_FIELD_REWARD: return e->a.reward;
        case B200RL_FIELD_TERMINAL: case B200RL_FIELD_FLAGS: return e->a.flags;
        case B200RL_FIELD_T: return e->a.t;
        case B200RL_FIELD_RNG: return e->a.rng;
        case B200RL_FIELD_ACTION: return e->a.action;
        case B200RL_FIELD_EPISODE_RETURN: return e->a.ep_ret;
        case B200RL_FIELD_EPISODE_STATS: return e->a.stats;
    }
    return nullptr;
}

static int env_alloc(b200rl_env* e) {
    size_t N = (size_t)e->N;
    CUDA_TRY(cudaMalloc(&e->a.state, N * e->ns * e->tsize));
    if (e->kind == B200RL_ENV_PENDULUM || e->kind == B200RL_ENV_ACROBOT) CUDA_TRY(cudaMalloc(&e->a.obs, N * e->nobs * e->tsize));
    else e->a.obs = e->a.state;
    CUDA_TRY(cudaMalloc(&e->a.reward, N * e->tsize));
    CUDA_TRY(cudaMalloc(&e->a.flags, N));
    CUDA_TRY(cudaMalloc(&e->a.t, N * 4));
    CUDA_TRY(cudaMalloc(&e->a.rng, N * 32));
    CUDA_TRY(cudaMalloc(&e->a.action, N * 8));
    CUDA_TRY(cudaMalloc(&e->a.ep_ret, N * 4));
    CUDA_TRY(cudaMalloc(&e->a.stats, 4 * sizeof(double)));
    CUDA_TRY(cudaMalloc(&e->a.err, sizeof(int)));
    cudaStream_t st = e->ctx->stream;
    CUDA_TRY(cudaMemsetAsync(e->a.state, 0, N * e->ns * e->tsize, st));
    if (e->a.obs != e->a.state) CUDA_TRY(cudaMemsetAsync(e->a.obs, 0, N * e->nobs * e->tsize, st));
    CUDA_TRY(cudaMemsetAsync(e->a.reward, 0, N * e->tsize, st));
    CUDA_TRY(cudaMemsetAsync(e->a.flags, 0, N, st));
    CUDA_TRY(cudaMemsetAsync(e->a.t, 0, N * 4, st));
    CUDA_TRY(cudaMemsetAsync(e->a.action, 0, N * 8, st));
    CUDA_TRY(cudaMemsetAsync(e->a.ep_ret, 0, N * 4, st));
    CUDA_TRY(cudaMemsetAsync(e->a.stats, 0, 4 * sizeof(double), st));
    CUDA_TRY(cudaMemsetAsync(e->a.err, 0, sizeof(int), st));
    e->a.traj_reward = nullptr;
    e->a.traj_terminal = nullptr;
    return B200RL_OK;
}

extern "C" {

int b200rl_env_create(b200rl_ctx* ctx, int kind, int dtype, int64_t n_envs, const void* params,
                      const uint64_t* rng_state, b200rl_env** out) {
    TRY(ctx_bind(ctx));
    REQUIRE(out && rng_state, B200RL_ERR_INVALID, "null out / rng_state");
    REQUIRE(n_envs > 0, B200RL_ERR_INVALID, "n_envs must be positive");
    REQUIRE(dtype == B200RL_F32 || dtype == B200RL_F64, B200RL_ERR_INVALID, "dtype must be B200RL_F32 or B200RL_F64");
    b200rl_env* e = new b200rl_env();
    memset(&e->a, 0, sizeof e->a);
    bool cont_kind = kind == B200RL_ENV_CARTPOLE_CONTINUOUS || kind == B200RL_ENV_MOUNTAINCAR_CONTINUOUS;
    if (kind == B200RL_ENV_CARTPOLE_CONTINUOUS && dtype != B200RL_F32) { delete e; REQUIRE(false, B200RL_ERR_UNSUPPORTED, "CartPoleEnv(continuous = true) is Float32 only"); }
    if (kind == B200RL_ENV_CARTPOLE_CONTINUOUS) kind = B200RL_ENV_CARTPOLE;
    if (kind == B200RL_ENV_MOUNTAINCAR_CONTINUOUS) kind = B200RL_ENV_MOUNTAINCAR;
    e->ctx = ctx; e->kind = kind; e->dtype = dtype; e->N = n_envs; e->continuous = cont_kind;
    e->tsize = dtype == B200RL_F64 ? 8 : 4;
    e->steps_launched = 0;
    if (kind == B200RL_ENV_CARTPOLE) {
        b200rl_cartpole_params d;
        if (params) d = *(const b200rl_cartpole_params*)params;
        else if (dtype == B200RL_F64)
            d = b200rl_cartpole_params{9.8, 1.0, 0.1, 1.0 + 0.1, 0.5, 0.1 * 0.5, 10.0, 0.02, 12.0 * JLD_PI / 180, 2.4, 200};
        else
            d = b200rl_cartpole_params{(float)9.8, 1.0, (float)0.1, (float)(1.0 + 0.1), 0.5, (float)(0.1 * 0.5), 10.0, (float)0.02,
                                       (float)(12.0 * JLD_PI / 180), (float)2.4, 200};
        e->ns = 4; e->nobs = 4;
        if (dtype == B200RL_F64)
            e->p.cp64 = CartPoleD<double>::P{d.gravity, d.totalmass, d.masspole, d.halflength, d.polemasslength, d.forcemag, d.dt,
                                              d.thetathreshold, d.xthreshold, (int)d.max_steps};
        else
            e->p.cp32 = CartPoleD<float>::P{(float)d.gravity, (float)d.totalmass, (float)d.masspole, (float)d.halflength,
                                             (float)d.polemasslength, (float)d.forcemag, (float)d.dt, (float)d.thetathreshold,
                                             (float)d.xthreshold, (int)d.max_steps};
    } else if (kind == B200RL_ENV_PENDULUM) {
        b200rl_pendulum_params d = params ? *(const b200rl_pendulum_params*)params
                                          : b200rl_pendulum_params{8, 2, 10, 1, 1, (float)0.05, 200, 3, 1};
        REQUIRE(d.continuous || d.n_actions >= 2, B200RL_ERR_INVALID, "n_actions must be >= 2");
        e->ns = 2; e->nobs = 3; e->continuous = d.continuous != 0;
        if (dtype == B200RL_F64) {   // PendulumEnv() default T = Float64 (PendulumEnv.jl:42): dt = Float64(0.05) unless the caller says otherwise
            if (!params) d.dt = 0.05;
            e->p.pend64 = PendPT<double>{d.max_speed, d.max_torque, d.g, d.m, d.l, d.dt, (int)d.max_steps, (int)d.n_actions};
        } else {
            e->p.pend = PendP{(float)d.max_speed, (float)d.max_torque, (float)d.g, (float)d.m, (float)d.l, (float)d.dt,
                              (int)d.max_steps, (int)d.n_actions};
        }
    } else if (kind == B200RL_ENV_MOUNTAINCAR) {
        // ContinuousMountainCarEnv defaults: goal_pos = 0.45, power = 0.0015 (MountainCarEnv.jl:73-74)
        b200rl_mountaincar_params d = params ? *(const b200rl_mountaincar_params*)params
                                      : cont_kind ? b200rl_mountaincar_params{(float)-1.2, (float)0.6, (float)0.07, (float)0.45, 0.0,
                                                                              (float)0.0015, (float)0.0025, 200}
                                                  : b200rl_mountaincar_params{(float)-1.2, (float)0.6, (float)0.07, (float)0.5, 0.0,
                                                                              (float)0.001, (float)0.0025, 200};
        e->ns = 2; e->nobs = 2;
        if (dtype == B200RL_F64) {   // MountainCarEnv() default T = Float64 (MountainCarEnv.jl:67): the Float64 literals of :19-29
            if (!params) d = cont_kind ? b200rl_mountaincar_params{-1.2, 0.6, 0.07, 0.45, 0.0, 0.0015, 0.0025, 200}
                                       : b200rl_mountaincar_params{-1.2, 0.6, 0.07, 0.5, 0.0, 0.001, 0.0025, 200};
            e->p.mc64 = MountainCarPT<double>{d.min_pos, d.max_pos, d.max_speed, d.goal_pos, d.goal_velocity, d.power, d.gravity, (int)d.max_steps};
        } else {
            e->p.mc = MountainCarD<false>::P{(float)d.min_pos, (float)d.max_pos, (float)d.max_speed, (float)d.goal_pos, (float)d.goal_velocity,
                                             (float)d.power, (float)d.gravity, (int)d.max_steps};
        }
    } else if (kind == B200RL_ENV_ACROBOT) {
        if (dtype != B200RL_F64) { delete e; REQUIRE(false, B200RL_ERR_UNSUPPORTED, "AcrobotEnv is Float64 only (the reference constructor's default T)"); }
        b200rl_acrobot_params d = params ? *(const b200rl_acrobot_params*)params
                                         : b200rl_acrobot_params{1.0, 1.0, 1.0, 1.0, 0.5, 0.5, 1.0, 0.0, 4 * JLD_PI, 9 * JLD_PI, 9.8, 0.2, 200, 1};
        if (d.max_torque_noise != 0.0) { delete e; REQUIRE(false, B200RL_ERR_UNSUPPORTED, "AcrobotEnv: max_torque_noise > 0 is not supported"); }
        e->ns = 4; e->nobs = 6;
        e->p.acro = AcrobotP{d.link_length_a, d.link_length_b, d.link_mass_a, d.link_mass_b, d.link_com_pos_a, d.link_com_pos_b, d.link_moi,
                             d.max_torque_noise, d.max_vel_a, d.max_vel_b, d.g, d.dt, (int)d.max_steps, (int)d.book};
    } else {
        delete e;
        REQUIRE(false, B200RL_ERR_INVALID, "unknown env kind");
    }
    e->asize = (e->continuous && dtype == B200RL_F64) ? 8 : 4;
    int s = env_alloc(e);
    if (s != B200RL_OK) { b200rl_env_destroy(e); return s; }
    CUDA_TRY(cudaMemcpyAsync(e->a.rng, rng_state, (size_t)n_envs * 32, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));  // rng_state is borrowed only for this call
    s = dispatch_reset(e, 1);  // the reference constructors call reset!(env) once
    if (s != B200RL_OK) { b200rl_env_destroy(e); return s; }
    *out = e;
    return B200RL_OK;
}

int b200rl_env_destroy(b200rl_env* e) {
    if (!e) return B200RL_OK;
    cudaSetDevice(e->ctx->device);
    cudaStreamSynchronize(e->ctx->stream);
    cudaFree(e->a.state);
    if (e->a.obs != e->a.state) cudaFree(e->a.obs);
    cudaFree(e->a.reward); cudaFree(e->a.flags); cudaFree(e->a.t); cudaFree(e->a.rng); cudaFree(e->a.action);
    cudaFree(e->a.ep_ret); cudaFree(e->a.stats); cudaFree(e->a.err);
    delete e;
    return B200RL_OK;
}

int b200rl_env_copy(b200rl_env* src, b200rl_env** out) {
    REQUIRE(src && out, B200RL_ERR_INVALID, "null handle");
    TRY(ctx_bind(src->ctx));
    b200rl_env* e = new b200rl_env(*src);
    memset(&e->a, 0, sizeof e->a);
    e->a.max_timeout = src->a.max_timeout;
    int s = env_alloc(e);
    if (s != B200RL_OK) { b200rl_env_destroy(e); return s; }
    cudaStream_t st = src->ctx->stream;
    for (int f : {B200RL_FIELD_STATE, B200RL_FIELD_REWARD, B200RL_FIELD_FLAGS, B200RL_FIELD_T, B200RL_FIELD_RNG, B200RL_FIELD_ACTION})
        CUDA_TRY(cudaMemcpyAsync(field_ptr(e, f), field_ptr(src, f), field_bytes(src, f), cudaMemcpyDeviceToDevice, st));
    if (e->a.obs != e->a.state)
        CUDA_TRY(cudaMemcpyAsync(e->a.obs, src->a.obs, field_bytes(src, B200RL_FIELD_OBS), cudaMemcpyDeviceToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(e->a.ep_ret, src->a.ep_ret, (size_t)src->N * 4, cudaMemcpyDeviceToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(e->a.stats, src->a.stats, 4 * sizeof(double), cudaMemcpyDeviceToDevice, st));
    *out = e;
    return B200RL_OK;
}

int b200rl_env_seed(b200rl_env* e, const uint64_t* rng_state) {
    REQUIRE(e && rng_state, B200RL_ERR_INVALID, "null argument");
    TRY(ctx_bind(e->ctx));
    CUDA_TRY(cudaMemcpyAsync(e->a.rng, rng_state, (size_t)e->N * 32, cudaMemcpyHostToDevice, e->ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(e->ctx->stream));
    return B200RL_OK;
}

int b200rl_env_reset(b200rl_env* e, int force_all) {
    REQUIRE(e, B200RL_ERR_INVALID, "null env");
    TRY(ctx_bind(e->ctx));
    return dispatch_reset(e, force_all);
}

int b200rl_env_step(b200rl_env* e, const void* actions, int actions_on_device, int auto_reset) {
    REQUIRE(e && actions, B200RL_ERR_INVALID, "null argument");
    TRY(ctx_bind(e->ctx));
    const void* dact = actions;
    if (actions_on_device != 1) {   // 0: pageable / borrowed host buffer, 2: pinned host buffer that stays untouched until the next sync
        void* stage;
        TRY(ctx_scratch(e->ctx, (size_t)e->N * e->asize, &stage));
        CUDA_TRY(cudaMemcpyAsync(stage, actions, (size_t)e->N * e->asize, cudaMemcpyHostToDevice, e->ctx->stream));
        dact = stage;
    }
    e->steps_launched += 1;
    TRY(dispatch_step(e, dact, false, auto_reset != 0));
    if (actions_on_device == 0) CUDA_TRY(cudaStreamSynchronize(e->ctx->stream));  // host buffer is borrowed for this call only
    return B200RL_OK;
}

int b200rl_env_set_max_timeout(b200rl_env* e, int64_t max_t) {
    REQUIRE(e, B200RL_ERR_INVALID, "null env");
    REQUIRE(max_t >= 0 && max_t < (1ll << 31), B200RL_ERR_INVALID, "max_t out of range");
    e->a.max_timeout = (int)max_t;
    return B200RL_OK;
}

int b200rl_env_step_random(b200rl_env* e, int auto_reset) {
    REQUIRE(e, B200RL_ERR_INVALID, "null env");
    REQUIRE(!e->continuous, B200RL_ERR_UNSUPPORTED,
            "RandomPolicy on a continuous interval (DomainSets sampler) is not restated; use a discrete-action env");
    TRY(ctx_bind(e->ctx));
    e->steps_launched += 1;
    return dispatch_step(e, nullptr, true, auto_reset != 0);
}

int b200rl_env_get(b200rl_env* e, int field, void* host_dst, size_t bytes) {
    REQUIRE(e && host_dst, B200RL_ERR_INVALID, "null argument");
    TRY(ctx_bind(e->ctx));
    size_t need = field_bytes(e, field);
    REQUIRE(need != 0, B200RL_ERR_INVALID, "unknown field");
    REQUIRE(bytes >= need, B200RL_ERR_INVALID, "destination too small");
    CUDA_TRY(cudaMemcpyAsync(host_dst, field_ptr(e, field), need, cudaMemcpyDeviceToHost, e->ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(e->ctx->stream));
    if (field == B200RL_FIELD_TERMINAL) {
        uint8_t* p = (uint8_t*)host_dst;
        for (size_t i = 0; i < need; ++i) p[i] &= 1;
    }
    if (field == B200RL_FIELD_EPISODE_STATS) ((double*)host_dst)[3] = (double)e->steps_launched * (double)e->N;   // host-side counter
    return B200RL_OK;
}

int b200rl_env_set(b200rl_env* e, int field, const void* host_src, size_t bytes) {
    REQUIRE(e && host_src, B200RL_ERR_INVALID, "null argument");
    TRY(ctx_bind(e->ctx));
    size_t need = field_bytes(e, field);
    REQUIRE(need != 0 && field != B200RL_FIELD_TERMINAL, B200RL_ERR_INVALID, "field not settable (TERMINAL is bit 0 of FLAGS)");
    REQUIRE(bytes >= need, B200RL_ERR_INVALID, "source too small");
    CUDA_TRY(cudaMemcpyAsync(field_ptr(e, field), host_src, need, cudaMemcpyHostToDevice, e->ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(e->ctx->stream));
    if (field == B200RL_FIELD_EPISODE_STATS) e->steps_launched = (uint64_t)(((const double*)host_src)[3] / (double)e->N + 0.5);
    return B200RL_OK;
}

int b200rl_env_ptr(b200rl_env* e, int field, void** dptr_out) {
    REQUIRE(e && dptr_out, B200RL_ERR_INVALID, "null argument");
    void* p = field_ptr(e, field);
    REQUIRE(p, B200RL_ERR_INVALID, "unknown field");
    *dptr_out = p;
    return B200RL_OK;
}

int b200rl_env_check(b200rl_env* e) {
    REQUIRE(e, B200RL_ERR_INVALID, "null env");
    TRY(ctx_bind(e->ctx));
    int flag = 0;
    CUDA_TRY(cudaMemcpyAsync(&flag, e->a.err, sizeof flag, cudaMemcpyDeviceToHost, e->ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(e->ctx->stream));
    if (flag) {
        CUDA_TRY(cudaMemsetAsync(e->a.err, 0, sizeof(int), e->ctx->stream));
        b200rl_set_error("b200rl_env_step: an action outside action_space(env) was passed (the reference asserts `a in action_space(env)`)");
        return B200RL_ERR_ACTION;
    }
    return B200RL_OK;
}

int b200rl_env_episode_stats(b200rl_env* e, double* out4, int reset_after) {
    REQUIRE(e && out4, B200RL_ERR_INVALID, "null argument");
    TRY(ctx_bind(e->ctx));
    CUDA_TRY(cudaMemcpyAsync(out4, e->a.stats, 4 * sizeof(double), cudaMemcpyDeviceToHost, e->ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(e->ctx->stream));
    out4[3] = (double)e->steps_launched * (double)e->N;
    if (reset_after) {
        CUDA_TRY(cudaMemsetAsync(e->a.stats, 0, 4 * sizeof(double), e->ctx->stream));
        e->steps_launched = 0;
    }
    return B200RL_OK;
}

}  // extern "C"

// internal hooks for other translation units (fused consumers)
int b200rl_env_internal_set_traj_targets(b200rl_env* e, void* reward_col, uint8_t* terminal_col) {
    e->a.traj_reward = reward_col;
    e->a.traj_terminal = terminal_col;
    return B200RL_OK;
}
int b200rl_env_internal_view(b200rl_env* e, envdev::EnvView* out) {
    REQUIRE(e && out, B200RL_ERR_INVALID, "null argument");
    out->kind = e->kind; out->dtype = e->dtype; out->continuous = e->continuous ? 1 : 0; out->N = e->N; out->a = e->a;
    static_assert(sizeof(out->p) == sizeof(e->p), "params union");
    memcpy(&out->p, &e->p, sizeof out->p);
    return B200RL_OK;
}
void b200rl_env_internal_add_steps(b200rl_env* e, uint64_t n) { e->steps_launched += n; }
int b200rl_env_internal_max_timeout(const b200rl_env* e) { return e->a.max_timeout; }
int b200rl_env_internal_dtype(const b200rl_env* e) { return e->dtype; }
int64_t b200rl_env_internal_n(const b200rl_env* e) { return e->N; }
int b200rl_env_internal_kind(const b200rl_env* e) { return e->kind; }
int b200rl_env_internal_nobs(const b200rl_env* e) { return e->nobs; }
b200rl_ctx* b200rl_env_internal_ctx(const b200rl_env* e) { return e->ctx; }
bool b200rl_env_internal_continuous(const b200rl_env* e) { return e->continuous; }
