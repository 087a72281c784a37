// internal.h — functions one translation unit of libb200rl.so provides to another (not part of the C ABI).  Included by the
// defining and the using files alike, so the compiler checks every definition against its declaration.
#pragma once
#include "common.cuh"

namespace envdev { struct EnvView; }

// env.cu: hooks for the fused consumers (agent, fused rollout)
int b200rl_env_internal_set_traj_targets(b200rl_env* e, void* reward_col, uint8_t* terminal_col);
int b200rl_env_internal_view(b200rl_env* e, envdev::EnvView* out);
void b200rl_env_internal_add_steps(b200rl_env* e, uint64_t n);
int b200rl_env_internal_max_timeout(const b200rl_env* e);
int b200rl_env_internal_dtype(const b200rl_env* e);
int64_t b200rl_env_internal_n(const b200rl_env* e);
int b200rl_env_internal_kind(const b200rl_env* e);
int b200rl_env_internal_nobs(const b200rl_env* e);
b200rl_ctx* b200rl_env_internal_ctx(const b200rl_env* e);
bool b200rl_env_internal_continuous(const b200rl_env* e);

// traj.cu: the batch gathered by the last b200rl_traj_sample, and the priority write-back
struct TrajBatchView { const float* s; const int32_t* a; const float* r; const uint8_t* t; const float* s2; const float* w; int64_t B; int ns; };
TrajBatchView b200rl_traj_internal_batch(b200rl_traj* t);
bool b200rl_traj_internal_prioritized(b200rl_traj* t);
b200rl_ctx* b200rl_traj_internal_ctx(b200rl_traj* t);
int64_t b200rl_traj_internal_lanes(b200rl_traj* t);
int b200rl_traj_internal_priority_from_td(b200rl_traj* t, const float* td_dev, float eps, float alpha);

// returns.cu: fused GAE of the (N, T) rollout (partials: b200rl_gae_fused_partials_count(S) doubles)
int b200rl_gae_fused_internal(b200rl_ctx* ctx, float* adv, float* ret, const float* r, const float* v, const uint8_t* term, float gamma,
                              float lambda, int64_t S, int64_t n_time, double* partials, float* norm2);
int b200rl_gae_fused_partials_count(int64_t S);

// comm.cu
int b200rl_comm_allreduce_internal(b200rl_ctx* ctx, void* buf, int64_t n, int is_double);
void b200rl_comm_destroy_internal(b200rl_ctx* ctx);
