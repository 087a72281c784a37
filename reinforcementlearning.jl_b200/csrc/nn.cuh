// nn.cuh — shared declarations of the learner kernels (nn.cu) for algo.cu.
//
// Network = Dense(in,H,act) -> Dense(H,H,act) -> head(s); parameters flat in
// Flux.destructure order, weights (out,in) column-major (W[o + out*i]):
//   W1 (H x in), b1 (H), W2 (H x H), b2 (H), then
//   single head:     W3 (n_out x H), b3 (n_out)                      [categorical logits / value / Q]
//   gaussian heads:  Wmu (1 x H), bmu (1), Wsig (1 x H), bsig (1)    [GaussianNetwork mu / sigma, 1-d action]
// (ActorCritic RLCore/src/utils/networks.jl:15-20, GaussianNetwork :44-116.)
#pragma once
#include "common.cuh"

constexpr int kInMax = 4;    // observation width <= 4 (CartPole 4, Pendulum 3, MountainCar 2)
constexpr int kOutMax = 4;   // head width <= 4

enum { B200RL_ACT_RELU = 0, B200RL_ACT_TANH = 1 };

struct MlpDesc {
    int in, H, act, nout, heads2;  // heads2: two 1-wide heads (gaussian mu / sigma)
    __host__ __device__ int64_t nparams() const { return (int64_t)H * in + H + (int64_t)H * H + H + (int64_t)nout * H + nout; }
};

struct AcHyper {  // scalars of the actor-critic losses (SURVEY Appendix B)
    float clip_range, w_actor, w_critic, w_entropy, min_sigma, max_sigma;
    int normalize_adv;
    int algo;  // 0 PPO clipped surrogate, 1 A2C (logp * advantage)
};

// One minibatch of the on-policy update: sample j is flat index perm(j) into the rollout
// arrays (states (ns, total) column-major; actions / logp_old / adv / ret (total)).
struct AcBatch {
    const float* states; int ns;
    const void* actions;        // int32 (1-based) or float
    const float* logp_old; const float* adv; const float* ret;
    const int32_t* idx;         // explicit permutation slice, or null ->
    uint32_t perm_n, perm_key, perm_offset;  // ... Feistel permutation of [0, perm_n), slice start
    const uint32_t* perm_epoch; // device update counter (may be null): the key actually used is perm_key + *perm_epoch * 1000003
    const float4* rec;          // packed 32-byte rollout records (may be null): rec[2j] = state (zero padded), rec[2j+1] =
                                // {action bits, logp_old, advantage, return} — one DRAM sector per gathered sample instead of five
    int64_t B;                  // samples in this minibatch (local)
    float inv_B;                // 1 / (global minibatch size)  — gradients are sums * inv_B
    const float* norm2;         // device {mean, inv_std} for advantage normalisation
};

// Optimiser state and hyper-parameters of one optimiser step (reduce the per-CTA partials -> [NVLink peer exchange] -> global norm ->
// clip_by_global_norm! -> Adam), whichever kernels run it (opt_path.h).
struct OptStep {
    float* params; float* grad; float* m; float* v; float* beta_t;
    float* loss_out4; float* stats_row; float* gnorm_out;     // each may be null
    double* cta_sumsq;            // >= 148 doubles
    unsigned int* counter;        // 4 zero-initialised uints (self-resetting grid barriers)
    unsigned int* tick;           // may be null: device update counter incremented once by the launch
    unsigned int* seq_ptr;        // gradient-exchange sequence number (sharded run)
    float max_norm, lr, b1, b2, eps;
    P2PTable tab;                 // nranks <= 1: no peer exchange
};
// K7 + optimiser step in ONE launch (OPT_FUSED_TAIL): the step runs in the tail of the tensor-core K7 behind two grid barriers (the
// 148 persistent CTAs are co-resident) instead of a second kernel (~14-20 us of launch, L2 round trips and barrier per optimiser
// step).  Returns the number of gradient partials (> 0) like nn_ac_loss_grad, or a negative status.
int nn_ac_loss_grad_step(b200rl_ctx* ctx, const MlpDesc& actor, const MlpDesc& critic, const AcHyper& hp, const AcBatch& b, float* partial,
                         float* loss_partial, const OptStep& st);

#ifdef __CUDACC__
__device__ __forceinline__ uint32_t ac_perm_key(const AcBatch& b) { return b.perm_key + (b.perm_epoch ? *b.perm_epoch * 1000003u : 0u); }
#endif
int nn_grid_ctas(b200rl_ctx* ctx, int H);  // persistent CTAs per role
int nn_dqn_max_partials(b200rl_ctx* ctx, int H);
// forward (rollout inference).  obs (in, N) column-major.  Any output may be null.
int nn_policy_act(b200rl_ctx* ctx, const MlpDesc& actor, const MlpDesc& critic, const float* params, const AcHyper& hp,
                  const float* obs, int64_t N, unsigned long long* rng, void* action_out, float* logp_out, float* value_out,
                  float* head_out /* (nout, N) raw head outputs, for tests */, float* state_copy /* (in, N) */);
int nn_mlp_forward(b200rl_ctx* ctx, const MlpDesc& net, const float* params, const float* obs, int64_t N, float* out /* (nout, N) */);
// loss + backward: writes per-CTA partial gradients/losses; nn_reduce sums them in CTA order.
// Returns the number of gradient partials written (> 0; loss rows = 2x that) or a negative status.
int nn_ac_loss_grad(b200rl_ctx* ctx, const MlpDesc& actor, const MlpDesc& critic, const float* params, const AcHyper& hp,
                    const AcBatch& b, float* partial /* [ctas][np] */, float* loss_partial /* [2*ctas][4] */);
int nn_ac_partial_rows(b200rl_ctx* ctx, const MlpDesc& actor, const MlpDesc& critic, const AcHyper& hp, int64_t B);   // what nn_ac_loss_grad returns
bool nn_fused_step_enabled();   // B200RL_FUSED_STEP / b200rl_set_fused_step
bool nn_tc_fused_tail_fits(b200rl_ctx* ctx, const MlpDesc& actor, const AcHyper& hp, int64_t B, int64_t np);   // opt_fused_tail_fits for K7
int nn_reduce_partials(b200rl_ctx* ctx, const float* partial, int n_partials, int64_t np, float* grad, const float* loss_partial,
                       int n_loss_partials, float* loss_out4);
// clip_by_global_norm! + Optimisers Adam on a flat gradient (single CTA, deterministic)
int nn_clip_adam(b200rl_ctx* ctx, float* params, float* grad, float* m, float* v, float* beta_t /* device [2] */, int64_t np,
                 float max_grad_norm, float lr, float b1, float b2, float eps, float grad_scale, float* gnorm_out /* device */);
// fused single-launch variant (OPT_ONE_KERNEL, OPT_ONE_KERNEL_XCHG when st.tab has peers; st.stats_row receives {4 loss sums,
// grad norm}): needs all ceil(np / 256) CTAs co-resident
int nn_reduce_clip_adam(b200rl_ctx* ctx, const float* partial, int n_partials, int64_t np, const float* loss_partial, int n_loss, const OptStep& st);
int nn_target_sync(b200rl_ctx* ctx, float* target, const float* model, int64_t np, float rho);
// DQN: TD loss + backward on a gathered batch (device arrays s (in,B), a, r, t, s2, w)
int nn_dqn_loss_grad(b200rl_ctx* ctx, const MlpDesc& q, const float* params, const float* target, const float* s, const int32_t* a,
                     const float* r, const uint8_t* t, const float* s2, const float* w, int64_t B, float inv_B, float gamma, int huber,
                     int double_dqn, float* partial, float* loss_partial, float* td_out);
int nn_q_act(b200rl_ctx* ctx, const MlpDesc& q, const float* params, const float* obs, int64_t N, unsigned long long* rng, float epsilon,
             int32_t* action_out, float* q_out);
int nn_q_explore(b200rl_ctx* ctx, const MlpDesc& q, const float* params, const float* obs, int64_t N, unsigned long long* rng,
                 const b200rl_explorer& ex, int32_t* action_out, float* q_out);

// tensor-core (tcgen05) variants, nn_tc.cu.  Used for H = 64 unless disabled (B200RL_TC=0 or b200rl_set_tensor_cores(0)).
bool nn_tc_enabled();
bool nn_tc_supported(const MlpDesc& d);
int nn_tc_forward(b200rl_ctx* ctx, int grid, const MlpDesc& actor, const MlpDesc& critic, const float* params, const AcHyper& hp, int mode,
                  const float* obs, int64_t N, unsigned long long* rng, void* action_out, float* logp_out, float* value_out, float* head_out,
                  float* state_copy);
// fused rollout (fwd_tc.cu): nsteps x {policy inference, env step, transition push} in one launch; B200RL_ERR_UNSUPPORTED =
// outside the fused envelope, step through nn_policy_act + b200rl_env_step instead
struct b200rl_env;
int nn_tc_rollout(b200rl_ctx* ctx, b200rl_env* env, const MlpDesc& actor, const MlpDesc& critic, const float* params, const AcHyper& hp,
                  unsigned long long* policy_rng, int t0, int nsteps, int T, int final_bootstrap, float* states, void* actions, float* logp,
                  float* values, float* rewards, uint8_t* terminals);
bool nn_tc_bwd_supported(const MlpDesc& actor, const MlpDesc& critic);
int nn_tc_partial_rows(int grid, const MlpDesc& actor, const AcHyper& hp, int64_t B);   // gradient-partial rows the tensor-core K7 writes with `grid` CTAs
int nn_tc_ac_loss_grad(b200rl_ctx* ctx, int grid, const MlpDesc& actor, const MlpDesc& critic, const float* params, const AcHyper& hp,
                       const AcBatch& b, float* partial, float* loss_partial, int64_t np, const OptStep* step /* null: loss + backward only */);
