// fwd_tc.cu — K6 on tensor cores and the fused rollout kernel (K6 + K1 + K3 over a whole rollout in ONE launch).
//
//   forward_tc_kernel  : policy inference for one env batch (plan!): actor -> action + log-prob, critic -> value.
//   rollout_tc_kernel  : n_steps x { obs -> actor -> sample action -> critic -> value -> env step (+ fused auto-reset) ->
//                        write the transition into column t of the rollout tensors }.  A CTA owns up to two tiles of 128
//                        envs for the whole launch; their env state and both RNG streams stay in shared memory, the weights of
//                        both networks too.  Replaces 2 launches per env step (agent_base.jl:45-66 stage loop, run.jl:52-68).
//
// Both kernels are built from the same device functions (tc_fwd.cuh, env_device.cuh) and compiled with the env flags
// (-fmad=false): stepping through plan!/act! one launch at a time or through the fused rollout gives bit-identical results.
#include "common.cuh"
#include "env_device.cuh"
#include "internal.h"
#include "tc_fwd.cuh"

using namespace tcfwd;
using namespace envdev;

namespace {

struct SmemFwd {
    NetSm net;
    float X[kInMax * TM];                 // [i][s]
    float Zp[2 * kOutMax * TM];           // head partials [half][o][s]
    alignas(8) uint64_t bar;
    uint32_t tmem;
};

__device__ __forceinline__ void load_rng32(const unsigned long long* rng, int64_t i, unsigned long long (&s)[4]) {
    const ulonglong2* p = reinterpret_cast<const ulonglong2*>(rng + 4 * i);
    ulonglong2 a = p[0], b = p[1];
    s[0] = a.x; s[1] = a.y; s[2] = b.x; s[3] = b.y;
}
__device__ __forceinline__ void store_rng32(unsigned long long* rng, int64_t i, const unsigned long long (&s)[4]) {
    ulonglong2* p = reinterpret_cast<ulonglong2*>(rng + 4 * i);
    p[0] = make_ulonglong2(s[0], s[1]);
    p[1] = make_ulonglong2(s[2], s[3]);
}

// mode 0: actor-critic rollout step (CTA role = blockIdx & 1), mode 1: plain forward of `actor` -> head_out
template <int ACT>
__global__ void __launch_bounds__(NT, 2)
forward_tc_kernel(MlpDesc actor, MlpDesc critic, const float* __restrict__ params, AcHyper hp, int mode, const float* __restrict__ obs,
                  int64_t N, unsigned long long* __restrict__ rng, void* __restrict__ action_out, float* __restrict__ logp_out,
                  float* __restrict__ value_out, float* __restrict__ head_out, float* __restrict__ state_copy) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    SmemFwd& sm = *reinterpret_cast<SmemFwd*>(smem_raw);
    const int nroles = mode == 0 ? 2 : 1;
    const int role = mode == 0 ? (blockIdx.x & 1) : 0;
    const int cta = blockIdx.x / nroles, nctas = gridDim.x / nroles;
    const MlpDesc d = role ? critic : actor;
    const int64_t poff = role ? actor.nparams() : 0;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int q = warp & 3, c = warp >> 2;
    const int s = 32 * q + lane;
    load_net(sm.net, d, params + poff, (ACT >= 0 ? ACT : d.act) == B200RL_ACT_RELU && ACT >= 0 ? kScale : 1.0f);
    if (warp == 0) umma::tmem_alloc(&sm.tmem, TMEM_COLS);
    if (tid == 32) umma::mbar_init(&sm.bar, 1);
    umma::fence_proxy_async();
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = sm.tmem;
    const uint32_t tmem_lane = tmem + ((uint32_t)(32 * q) << 16);
    const int64_t ntiles = (N + TM - 1) / TM;
    uint32_t phase = 0;
    for (int64_t tile = cta; tile < ntiles; tile += nctas) {
        if (tid < TM) {
            int64_t i = tile * TM + tid;
            float x[kInMax] = {0.f, 0.f, 0.f, 0.f};
            if (i < N) {
                if (d.in == 4) {
                    float4 v4 = reinterpret_cast<const float4*>(obs)[i];
                    x[0] = v4.x; x[1] = v4.y; x[2] = v4.z; x[3] = v4.w;
                    if (state_copy && role == 0) reinterpret_cast<float4*>(state_copy)[i] = v4;
                } else {
#pragma unroll
                    for (int k = 0; k < kInMax; ++k) {
                        if (k < d.in) {
                            x[k] = obs[(int64_t)d.in * i + k];
                            if (state_copy && role == 0) state_copy[(int64_t)d.in * i + k] = x[k];
                        }
                    }
                }
            }
#pragma unroll
            for (int k = 0; k < kInMax; ++k) sm.X[k * TM + tid] = x[k];
        }
        __syncthreads();
        {
            float x[kInMax];
#pragma unroll
            for (int k = 0; k < kInMax; ++k) x[k] = sm.X[k * TM + s];
            layer1_to_tmem<ACT>(sm.net, d.act, x, c, tmem_lane);
        }
        umma::fence_before_sync();
        __syncthreads();
        if (tid == 0) {   // (elect.sync measured 3 % slower here, profiles/umma_pacing.py notes)
            umma::fence_after_sync();
            issue_gemm(tmem, sm.net);
            umma::commit(&sm.bar);
        }
        __syncwarp();
        umma::mbar_wait(&sm.bar, phase);
        phase ^= 1u;
        umma::fence_after_sync();
        {
            float zp[kOutMax];
            head_partials<ACT>(sm.net, d.act, c, tmem_lane, zp);
#pragma unroll
            for (int o = 0; o < kOutMax; ++o) sm.Zp[(c * kOutMax + o) * TM + s] = zp[o];
        }
        umma::fence_before_sync();     // TMEM reads done before the next tile's layer 1 / MMA overwrite A and D
        __syncthreads();
        if (tid < TM) {
            int64_t i = tile * TM + tid;
            if (i < N) {
                float z[kOutMax];
#pragma unroll
                for (int o = 0; o < kOutMax; ++o) z[o] = sm.net.b3[o] + sm.Zp[o * TM + tid] + sm.Zp[(kOutMax + o) * TM + tid];
                if (head_out && (mode == 1 || role == 0))
                    for (int o = 0; o < d.nout; ++o) head_out[(int64_t)d.nout * i + o] = z[o];
                if (mode == 0 && role == 1) {
                    if (value_out) value_out[i] = z[0];
                } else if (mode == 0) {
                    unsigned long long st[4];
                    load_rng32(rng, i, st);
                    float lp;
                    uint32_t a = sample_head(actor, hp, z, st, lp);
                    if (action_out) reinterpret_cast<uint32_t*>(action_out)[i] = a;
                    if (logp_out) logp_out[i] = lp;
                    store_rng32(rng, i, st);
                }
            }
        }
        __syncthreads();
    }
    umma::fence_before_sync();
    __syncthreads();
    if (warp == 0) umma::tmem_dealloc(tmem, TMEM_COLS);
}

// ---------------------------------------------------------------------------------------------------------------------
// fused rollout
constexpr int kSlots = 2;   // tiles of 128 envs a CTA keeps resident

template <class Env> struct SlotState {   // env state of one tile, one entry per env (owner thread = TMEM lane)
    typename Env::S st[TM];
    int t[TM];
    int flags[TM];
    float ep_ret[TM];
    float last_rew[TM];
    uint32_t last_act[TM];                 // env.action after the last act! (a reset may have redrawn it), raw bits
    unsigned long long erng[4 * TM];   // env stream  [word][env]
    unsigned long long prng[4 * TM];   // policy stream
};
template <class Env> struct SmemRoll {
    NetSm net[2];                          // actor, critic
    float X[kInMax * TM];
    float Zp[2][2 * kOutMax * TM];         // [net][half][o][s]
    SlotState<Env> slot[kSlots];
    float red_f[8];
    int red_i[8], red_l[8];
    alignas(8) uint64_t bar;
    uint32_t tmem;
};

struct RollArgs {
    MlpDesc actor, critic;
    const float* params;
    AcHyper hp;
    int64_t N;
    int t0, nsteps, T;          // rollout columns t0 .. t0 + nsteps - 1 of T
    int final_bootstrap;        // also write states[:, :, t0 + nsteps] and V of it (only when t0 + nsteps == T)
    float act_lo, act_hi;       // continuous actions: the env receives clamp(a, lo, hi), the rollout keeps a
    unsigned long long* policy_rng;   // (4, N)
    float* states;              // (NOBS, N, T + 1)
    void* actions;              // (N, T) int32 | f32
    float* logp;                // (N, T)
    float* values;              // (N, T + 1)
    float* rewards;             // (N, T)
    uint8_t* terminals;         // (N, T)
};

template <class Env, int ACT>
__global__ void __launch_bounds__(NT, 2) rollout_tc_kernel(RollArgs g, typename Env::P p, EnvArrays ea) {
    using act_t = typename Env::act_t;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    SmemRoll<Env>& sm = *reinterpret_cast<SmemRoll<Env>*>(smem_raw);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int q = warp & 3, c = warp >> 2;
    const int s = 32 * q + lane;
    const bool owner = c == 0;              // warps 0..3: thread s also owns env s of the tile
    const int cta = blockIdx.x, nctas = gridDim.x;
    const int64_t N = g.N;
    const int64_t ntiles = (N + TM - 1) / TM;
    load_net(sm.net[0], g.actor, g.params, ACT == B200RL_ACT_RELU ? kScale : 1.0f);
    load_net(sm.net[1], g.critic, g.params + g.actor.nparams(), ACT == B200RL_ACT_RELU ? kScale : 1.0f);
    if (warp == 0) umma::tmem_alloc(&sm.tmem, TMEM_COLS);
    if (tid == 32) umma::mbar_init(&sm.bar, 1);
    // resident env state
    int nslots = 0;
    for (int k = 0; k < kSlots; ++k)
        if ((int64_t)cta + (int64_t)k * nctas < ntiles) nslots = k + 1;
    if (owner) {
        for (int k = 0; k < nslots; ++k) {
            const int64_t i = ((int64_t)cta + (int64_t)k * nctas) * TM + s;
            SlotState<Env>& sl = sm.slot[k];
            if (i < N) {
                sl.st[s] = Env::load(ea.state, i);
                sl.t[s] = ea.t[i];
                sl.flags[s] = ea.flags[i];
                sl.ep_ret[s] = ea.ep_ret[i];
                Xo e = load_rng(ea.rng, i);
                sl.erng[s] = e.s0; sl.erng[TM + s] = e.s1; sl.erng[2 * TM + s] = e.s2; sl.erng[3 * TM + s] = e.s3;
                unsigned long long pr[4];
                load_rng32(g.policy_rng, i, pr);
                sl.prng[s] = pr[0]; sl.prng[TM + s] = pr[1]; sl.prng[2 * TM + s] = pr[2]; sl.prng[3 * TM + s] = pr[3];
            }
        }
    }
    umma::fence_proxy_async();
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = sm.tmem;
    const uint32_t tmem_lane = tmem + ((uint32_t)(32 * q) << 16);
    uint32_t phase = 0;
    // episode statistics of this thread's envs (device-side TotalRewardPerEpisode / BatchStepsPerEpisode, hooks.jl:146-231)
    int fin_cnt = 0, fin_len = 0;
    float fin_ret = 0.f;
    const int ns = Env::NOBS;
    const int nst = g.final_bootstrap ? g.nsteps + 1 : g.nsteps;
#pragma unroll 1
    for (int step = 0; step < nst; ++step) {
        const int t = g.t0 + step;
        const bool boot = step == g.nsteps;      // extra pass: V(s_T) only
#pragma unroll 1
        for (int k = 0; k < nslots; ++k) {
            SlotState<Env>& sl = sm.slot[k];
            const int64_t i = ((int64_t)cta + (int64_t)k * nctas) * TM + s;
            const bool live = i < N;
            // ---- observation of this step -> X (shared) and column t of the rollout states ------------------------
            if (owner) {
                float o[kInMax] = {0.f, 0.f, 0.f, 0.f};
                if (live) {
                    Env::observe(sl.st[s], o);
                    float* dst = g.states + ((size_t)N * ns) * (size_t)t + (size_t)ns * i;
                    if (ns == 4) *reinterpret_cast<float4*>(dst) = make_float4(o[0], o[1], o[2], o[3]);
                    else {
#pragma unroll
                        for (int j = 0; j < kInMax; ++j) if (j < ns) dst[j] = o[j];
                    }
                }
#pragma unroll
                for (int j = 0; j < kInMax; ++j) sm.X[j * TM + s] = o[j];
            }
            __syncthreads();
            float x[kInMax];
#pragma unroll
            for (int j = 0; j < kInMax; ++j) x[j] = sm.X[j * TM + s];
            uint32_t a_bits = 0;
            if (!boot) {
                // ---- actor ---------------------------------------------------------------------------------------
                layer1_to_tmem<ACT>(sm.net[0], g.actor.act, x, c, tmem_lane);
                umma::fence_before_sync();
                __syncthreads();
                if (tid == 0) {   // (elect.sync measured 3 % slower here, profiles/umma_pacing.py notes)
                    umma::fence_after_sync();
                    issue_gemm(tmem, sm.net[0]);
                    umma::commit(&sm.bar);
                }
                __syncwarp();
                umma::mbar_wait(&sm.bar, phase);
                phase ^= 1u;
                umma::fence_after_sync();
                {
                    float zp[kOutMax];
                    head_partials<ACT>(sm.net[0], g.actor.act, c, tmem_lane, zp);
#pragma unroll
                    for (int o = 0; o < kOutMax; ++o) sm.Zp[0][(c * kOutMax + o) * TM + s] = zp[o];
                }
                umma::fence_before_sync();
                __syncthreads();
            }
            // ---- critic GEMM in flight while the owner threads sample the action and step the env -----------------------
            layer1_to_tmem<ACT>(sm.net[1], g.critic.act, x, c, tmem_lane);
            umma::fence_before_sync();
            __syncthreads();
            if (tid == 0) {   // (elect.sync measured 3 % slower here, profiles/umma_pacing.py notes)
                umma::fence_after_sync();
                issue_gemm(tmem, sm.net[1]);
                umma::commit(&sm.bar);
            }
            __syncwarp();
            if (owner && live && !boot) {
                float z[kOutMax];
#pragma unroll
                for (int o = 0; o < kOutMax; ++o) z[o] = sm.net[0].b3[o] + sm.Zp[0][o * TM + s] + sm.Zp[0][(kOutMax + o) * TM + s];
                unsigned long long pr[4] = {sl.prng[s], sl.prng[TM + s], sl.prng[2 * TM + s], sl.prng[3 * TM + s]};
                float lp;
                a_bits = sample_head(g.actor, g.hp, z, pr, lp);
                sl.prng[s] = pr[0]; sl.prng[TM + s] = pr[1]; sl.prng[2 * TM + s] = pr[2]; sl.prng[3 * TM + s] = pr[3];
                reinterpret_cast<uint32_t*>(g.actions)[(size_t)N * t + i] = a_bits;
                g.logp[(size_t)N * t + i] = lp;
                // act!(env, a) + fused soft reset (MultiThreadEnv): same sequence as env_step_kernel<Env, false, true>
                act_t act;
                if (std::is_same<act_t, float>::value) act = (act_t)fminf(fmaxf(__uint_as_float(a_bits), g.act_lo), g.act_hi);
                else act = (act_t)(int32_t)a_bits;
                typename Env::S st = sl.st[s];
                int tt = sl.t[s];
                const int prev = sl.flags[s];
                bool done;
                float rew;
                Env::step(p, st, tt, act, done, rew);
                if (ea.max_timeout > 0 && tt + 1 > ea.max_timeout) done = true;
                float ret = sl.ep_ret[s] + rew;
                int f = done ? 1 : 0;
                if (done && !((prev & 1) && !(prev & 2))) { fin_cnt += 1; fin_ret += ret; fin_len += tt; }
                if (done) {
                    ret = 0.f;
                    Xo e{sl.erng[s], sl.erng[TM + s], sl.erng[2 * TM + s], sl.erng[3 * TM + s]};
                    Env::reset(p, st, e, act);
                    sl.erng[s] = e.s0; sl.erng[TM + s] = e.s1; sl.erng[2 * TM + s] = e.s2; sl.erng[3 * TM + s] = e.s3;
                    tt = 0;
                    f = 3;
                }
                sl.st[s] = st; sl.t[s] = tt; sl.flags[s] = f; sl.ep_ret[s] = ret;
                g.rewards[(size_t)N * t + i] = rew;
                g.terminals[(size_t)N * t + i] = done ? 1 : 0;
                sl.last_rew[s] = rew;
                { act_t tmp = act; uint32_t bits; memcpy(&bits, &tmp, 4); sl.last_act[s] = bits; }
            }
            umma::mbar_wait(&sm.bar, phase);
            phase ^= 1u;
            umma::fence_after_sync();
            {
                float zp[kOutMax];
                head_partials<ACT>(sm.net[1], g.critic.act, c, tmem_lane, zp);
                sm.Zp[1][(c * kOutMax) * TM + s] = zp[0];
            }
            umma::fence_before_sync();
            __syncthreads();
            if (owner && live) g.values[(size_t)N * t + i] = sm.net[1].b3[0] + sm.Zp[1][s] + sm.Zp[1][kOutMax * TM + s];
            // (the next pass's X / Zp writes are ordered behind this read by its first __syncthreads)
        }
    }
    // ---- write the env back ---------------------------------------------------------------------------------------
    if (owner) {
        for (int k = 0; k < nslots; ++k) {
            const int64_t i = ((int64_t)cta + (int64_t)k * nctas) * TM + s;
            SlotState<Env>& sl = sm.slot[k];
            if (i < N) {
                Env::store(ea.state, i, sl.st[s]);
                if (!Env::kObsIsState) Env::write_obs(ea.obs, i, N, sl.st[s]);
                ea.t[i] = sl.t[s];
                ea.flags[i] = (uint8_t)sl.flags[s];
                ea.ep_ret[i] = sl.ep_ret[s];
                store_rng(ea.rng, i, Xo{sl.erng[s], sl.erng[TM + s], sl.erng[2 * TM + s], sl.erng[3 * TM + s]});
                unsigned long long pr[4] = {sl.prng[s], sl.prng[TM + s], sl.prng[2 * TM + s], sl.prng[3 * TM + s]};
                store_rng32(g.policy_rng, i, pr);
                if (g.nsteps > 0) {
                    reinterpret_cast<float*>(ea.reward)[i] = sl.last_rew[s];
                    reinterpret_cast<uint32_t*>(ea.action)[i] = sl.last_act[s];
                }
            }
        }
    }
    // episode statistics: one atomicAdd triple per CTA
    {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            fin_cnt += __shfl_xor_sync(0xffffffffu, fin_cnt, o);
            fin_len += __shfl_xor_sync(0xffffffffu, fin_len, o);
            fin_ret += __shfl_xor_sync(0xffffffffu, fin_ret, o);
        }
        __syncthreads();
        if (lane == 0) { sm.red_i[warp] = fin_cnt; sm.red_f[warp] = fin_ret; sm.red_l[warp] = fin_len; }
        __syncthreads();
        if (tid == 0) {
            double cc = 0, rr = 0, ll = 0;
            for (int w = 0; w < NT / 32; ++w) { cc += sm.red_i[w]; rr += sm.red_f[w]; ll += sm.red_l[w]; }
            if (cc > 0) { atomicAdd(&ea.stats[0], cc); atomicAdd(&ea.stats[1], rr); atomicAdd(&ea.stats[2], ll); }
        }
    }
    umma::fence_before_sync();
    __syncthreads();
    if (warp == 0) umma::tmem_dealloc(tmem, TMEM_COLS);
}

template <class Env> int launch_rollout(b200rl_ctx* ctx, const RollArgs& g, const typename Env::P& p, const EnvArrays& ea) {
    const size_t smem = sizeof(SmemRoll<Env>) + 128;
    static unsigned long long attr_devices = 0;   // once per device: the attribute call is not free and may serialise with running kernels
    if (first_use_on_device(attr_devices, ctx->device)) {
        CUDA_TRY(cudaFuncSetAttribute(rollout_tc_kernel<Env, B200RL_ACT_RELU>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CUDA_TRY(cudaFuncSetAttribute(rollout_tc_kernel<Env, B200RL_ACT_TANH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
    const int64_t ntiles = (g.N + TM - 1) / TM;
    int grid = 2 * ctx->sm_count;
    if ((int64_t)grid > ntiles) grid = (int)ntiles;
    // the activation is a template parameter (nn_tc_rollout only comes here when both trunks share it)
    if (g.actor.act == B200RL_ACT_RELU) rollout_tc_kernel<Env, B200RL_ACT_RELU><<<grid, NT, smem, ctx->stream>>>(g, p, ea);
    else rollout_tc_kernel<Env, B200RL_ACT_TANH><<<grid, NT, smem, ctx->stream>>>(g, p, ea);
    LAUNCH_CHECK(ctx);
    return B200RL_OK;
}

}  // namespace

bool nn_tc_supported(const MlpDesc& d) { return d.H == 64 && d.in <= kInMax && d.nout <= kOutMax; }

int nn_tc_forward(b200rl_ctx* ctx, int grid, const MlpDesc& actor, const MlpDesc& critic, const float* params, const AcHyper& hp, int mode,
                  const float* obs, int64_t N, unsigned long long* rng, void* action_out, float* logp_out, float* value_out, float* head_out,
                  float* state_copy) {
    size_t smem = sizeof(SmemFwd) + 128;
    static unsigned long long attr_devices = 0;   // once per device
    if (first_use_on_device(attr_devices, ctx->device)) {
        CUDA_TRY(cudaFuncSetAttribute(forward_tc_kernel<B200RL_ACT_RELU>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CUDA_TRY(cudaFuncSetAttribute(forward_tc_kernel<B200RL_ACT_TANH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CUDA_TRY(cudaFuncSetAttribute(forward_tc_kernel<-1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
    const bool same = mode != 0 || actor.act == critic.act;   // mode 1 runs `actor` alone
    if (same && actor.act == B200RL_ACT_RELU)
        forward_tc_kernel<B200RL_ACT_RELU><<<grid, NT, smem, ctx->stream>>>(actor, critic, params, hp, mode, obs, N, rng, action_out, logp_out, value_out, head_out, state_copy);
    else if (same && actor.act == B200RL_ACT_TANH)
        forward_tc_kernel<B200RL_ACT_TANH><<<grid, NT, smem, ctx->stream>>>(actor, critic, params, hp, mode, obs, N, rng, action_out, logp_out, value_out, head_out, state_copy);
    else
        forward_tc_kernel<-1><<<grid, NT, smem, ctx->stream>>>(actor, critic, params, hp, mode, obs, N, rng, action_out, logp_out, value_out, head_out, state_copy);
    LAUNCH_CHECK(ctx);
    return B200RL_OK;
}

// Fused rollout of `nsteps` env steps starting at column t0.  Returns B200RL_ERR_UNSUPPORTED (without setting an error
// message the caller would surface) when the configuration is outside the fused kernel's envelope: the caller then steps
// through plan! / act! launches, which computes the same thing.
int nn_tc_rollout(b200rl_ctx* ctx, b200rl_env* env, const MlpDesc& actor, const MlpDesc& critic, const float* params, const AcHyper& hp,
                  unsigned long long* policy_rng, int t0, int nsteps, int T, int final_bootstrap, float* states, void* actions, float* logp,
                  float* values, float* rewards, uint8_t* terminals) {
    EnvView v;
    TRY(b200rl_env_internal_view(env, &v));
    if (!(nn_tc_supported(actor) && nn_tc_supported(critic)) || critic.nout != 1 || v.dtype != B200RL_F32) return B200RL_ERR_UNSUPPORTED;
    if (actor.act != critic.act) return B200RL_ERR_UNSUPPORTED;   // the fused kernel is compiled per activation (staged launches handle a mixed pair)
    const int64_t ntiles = (v.N + TM - 1) / TM;
    if (ntiles > (int64_t)kSlots * 2 * ctx->sm_count) return B200RL_ERR_UNSUPPORTED;
    if ((actor.heads2 != 0) != (v.continuous != 0)) return B200RL_ERR_UNSUPPORTED;   // Gaussian head <-> continuous action space
    RollArgs g{actor, critic, params, hp, v.N, t0, nsteps, T, final_bootstrap, -1.0f, 1.0f, policy_rng, states, actions, logp, values, rewards, terminals};
    int st = B200RL_ERR_UNSUPPORTED;
    switch (v.kind) {
        case B200RL_ENV_CARTPOLE:
            if (v.continuous) {
                CartPoleD<float, true>::P q;
                memcpy(&q, &v.p.cp32, sizeof q);
                st = launch_rollout<CartPoleD<float, true>>(ctx, g, q, v.a);
            } else {
                if (actor.nout != 2) return B200RL_ERR_UNSUPPORTED;
                st = launch_rollout<CartPoleD<float, false>>(ctx, g, v.p.cp32, v.a);
            }
            break;
        case B200RL_ENV_PENDULUM:
            if (v.continuous) {
                g.act_lo = -2.0f; g.act_hi = 2.0f;      // PendulumEnv.jl:73: action_space -2.0..2.0
                st = launch_rollout<PendulumD<true>>(ctx, g, v.p.pend, v.a);
            } else {
                if (actor.nout != v.p.pend.n_actions) return B200RL_ERR_UNSUPPORTED;
                st = launch_rollout<PendulumD<false>>(ctx, g, v.p.pend, v.a);
            }
            break;
        case B200RL_ENV_MOUNTAINCAR:
            if (v.continuous) {
                MountainCarD<true>::P q;
                memcpy(&q, &v.p.mc, sizeof q);
                st = launch_rollout<MountainCarD<true>>(ctx, g, q, v.a);
            } else {
                if (actor.nout != 3) return B200RL_ERR_UNSUPPORTED;
                st = launch_rollout<MountainCarD<false>>(ctx, g, v.p.mc, v.a);
            }
            break;
    }
    if (st == B200RL_OK) b200rl_env_internal_add_steps(env, (uint64_t)nsteps);
    return st;
}
