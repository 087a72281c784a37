// tests/hostdev/hostdev.cpp — TEST INFRASTRUCTURE.  The product's device headers compiled for the host (see cuda_runtime.h here) behind
// a flat C interface: Julia math kernels, Xoshiro samplers, env reset!/_step! per env, the minibatch permutation and the optimiser-step rule.  The control flow
// around the per-env primitives (auto-reset after a terminating step) restates env.cu's step kernel in the obvious serial way.
#include <cuda_runtime.h>

#include <vector>

#include "env_device.cuh"
#include "opt_path.h"
#include "perm.cuh"
#include "tc_split.h"

using namespace envdev;

extern "C" {

float hd_sin32(float x) { return jld::jsin(x); }
float hd_cos32(float x) { return jld::jcos(x); }
double hd_sin64(double x) { return jld::jsin(x); }
double hd_cos64(double x) { return jld::jcos(x); }
double hd_mod64(double x, double y) { return jld::jmod(x, y); }
uint32_t hd_perm_index(uint32_t q, uint32_t n, uint32_t key) { return b200perm::perm_index(q, n, key); }
int hd_tc_actor_ctas(int grid, int gaussian, int64_t ntiles) { return b200rl_tc_actor_ctas(grid, gaussian != 0, ntiles); }
// opt_path() with the fused tail's size limits evaluated by opt_fused_tail_fits(np, grid, rows, sm_count)
int hd_opt_path(int world, int p2p, int exclusive, int fused_step, int tc_bwd, int64_t np, int grid, int rows, int sm_count, int fits_inbox, int coresident) {
    return opt_path(OptPathIn{world, p2p != 0, exclusive != 0, fused_step != 0, tc_bwd != 0, opt_fused_tail_fits(np, grid, rows, sm_count), fits_inbox != 0,
                              coresident != 0});
}
int64_t hd_rand_oneto(uint64_t* s, uint64_t n) {
    jld::Xo g{s[0], s[1], s[2], s[3]};
    long long r = jld::rand_oneto(g, n);
    s[0] = g.s0; s[1] = g.s1; s[2] = g.s2; s[3] = g.s3;
    return r;
}

}  // extern "C"

namespace {
// One env object per index, stepped serially: t += 1 inside Env::step; a terminating step keeps its reward / terminal and (auto-reset)
// the state becomes the fresh episode's — exactly what the oracle's `step(actions, auto_reset = true)` and the kernel do.
template <class Env>
void run_env(const typename Env::P& p, int64_t n, int steps, uint64_t* rng, const void* actions, int random_policy, void* state_io,
             typename Env::real* reward_out, uint8_t* terminal_out, int32_t* t_io, void* action_out, int do_reset_first) {
    using act_t = typename Env::act_t;
    using real = typename Env::real;
    for (int64_t i = 0; i < n; ++i) {
        Xo g{rng[4 * i], rng[4 * i + 1], rng[4 * i + 2], rng[4 * i + 3]};
        typename Env::S s = Env::load(state_io, i);
        int t = t_io[i];
        act_t last = 0;
        if (do_reset_first) { Env::reset(p, s, g, last); t = 0; }
        real rew = 0;
        bool done = false;
        for (int k = 0; k < steps; ++k) {
            act_t a = random_policy ? Env::from_index(p, jld::rand_oneto(g, Env::n_random(p))) : reinterpret_cast<const act_t*>(actions)[(int64_t)k * n + i];
            Env::step(p, s, t, a, done, rew);
            last = a;
            reward_out[(int64_t)k * n + i] = rew;
            terminal_out[(int64_t)k * n + i] = done ? 1 : 0;
            if (done) { act_t dummy = 0; Env::reset(p, s, g, dummy); t = 0; }
        }
        Env::store(state_io, i, s);
        t_io[i] = t;
        if (action_out) reinterpret_cast<act_t*>(action_out)[i] = last;
        rng[4 * i] = g.s0; rng[4 * i + 1] = g.s1; rng[4 * i + 2] = g.s2; rng[4 * i + 3] = g.s3;
    }
}
}  // namespace

extern "C" {
// kind: 0 CartPole f32 | 1 Pendulum continuous | 2 MountainCar | 3 CartPole continuous f32 | 4 MountainCar continuous | 5 CartPole f64
//       | 6 Pendulum discrete | 7 Pendulum f64 continuous | 8 Pendulum f64 discrete | 9 MountainCar f64 | 10 MountainCar f64 continuous | 11 Acrobot f64.
//       q: the oracle's parameter vector (tests/oracle_lib.default_params layout).
// actions: (n, steps) column-major (int32 or float32 / ignored when random_policy); reward / terminal out: (n, steps).
int hd_env_run(int kind, const double* q, int64_t n, int steps, uint64_t* rng, const void* actions, int random_policy, void* state_io,
               void* reward_out, uint8_t* terminal_out, int32_t* t_io, void* action_out, int do_reset_first) {
    if (kind == 0 || kind == 3) {
        CartPoleD<float>::P p{(float)q[0], (float)q[3], (float)q[2], (float)q[4], (float)q[5], (float)q[6], (float)q[7], (float)q[8], (float)q[9], (int)q[10]};
        if (kind == 0) run_env<CartPoleD<float, false>>(p, n, steps, rng, actions, random_policy, state_io, (float*)reward_out, terminal_out, t_io, action_out, do_reset_first);
        else {
            CartPoleD<float, true>::P pc;
            static_assert(sizeof(pc) == sizeof(p), "same parameter struct");
            std::memcpy(&pc, &p, sizeof p);
            run_env<CartPoleD<float, true>>(pc, n, steps, rng, actions, 0, state_io, (float*)reward_out, terminal_out, t_io, action_out, do_reset_first);
        }
        return 0;
    }
    if (kind == 5) {
        CartPoleD<double>::P p{q[0], q[3], q[2], q[4], q[5], q[6], q[7], q[8], q[9], (int)q[10]};
        run_env<CartPoleD<double, false>>(p, n, steps, rng, actions, random_policy, state_io, (double*)reward_out, terminal_out, t_io, action_out, do_reset_first);
        return 0;
    }
    if (kind == 1 || kind == 6) {
        PendP p{(float)q[0], (float)q[1], (float)q[2], (float)q[3], (float)q[4], (float)q[5], (int)q[6], (int)q[7]};
        if (kind == 1) run_env<PendulumD<true>>(p, n, steps, rng, actions, 0, state_io, (float*)reward_out, terminal_out, t_io, action_out, do_reset_first);
        else run_env<PendulumD<false>>(p, n, steps, rng, actions, random_policy, state_io, (float*)reward_out, terminal_out, t_io, action_out, do_reset_first);
        return 0;
    }
    if (kind == 7 || kind == 8) {
        PendPT<double> p{q[0], q[1], q[2], q[3], q[4], q[5], (int)q[6], (int)q[7]};
        if (kind == 7) run_env<PendulumD<true, double>>(p, n, steps, rng, actions, 0, state_io, (double*)reward_out, terminal_out, t_io, action_out, do_reset_first);
        else run_env<PendulumD<false, double>>(p, n, steps, rng, actions, random_policy, state_io, (double*)reward_out, terminal_out, t_io, action_out, do_reset_first);
        return 0;
    }
    if (kind == 9 || kind == 10) {
        MountainCarPT<double> p{q[0], q[1], q[2], q[3], q[4], q[5], q[6], (int)q[7]};
        if (kind == 9) run_env<MountainCarD<false, double>>(p, n, steps, rng, actions, random_policy, state_io, (double*)reward_out, terminal_out, t_io, action_out, do_reset_first);
        else run_env<MountainCarD<true, double>>(p, n, steps, rng, actions, 0, state_io, (double*)reward_out, terminal_out, t_io, action_out, do_reset_first);
        return 0;
    }
    if (kind == 2 || kind == 4) {
        MountainCarD<false>::P p{(float)q[0], (float)q[1], (float)q[2], (float)q[3], (float)q[4], (float)q[5], (float)q[6], (int)q[7]};
        if (kind == 2) run_env<MountainCarD<false>>(p, n, steps, rng, actions, random_policy, state_io, (float*)reward_out, terminal_out, t_io, action_out, do_reset_first);
        else {
            MountainCarD<true>::P pc;
            std::memcpy(&pc, &p, sizeof p);
            run_env<MountainCarD<true>>(pc, n, steps, rng, actions, 0, state_io, (float*)reward_out, terminal_out, t_io, action_out, do_reset_first);
        }
        return 0;
    }
    if (kind == 11) {   // AcrobotEnv{Float64}
        AcrobotP p{q[0], q[1], q[2], q[3], q[4], q[5], q[6], q[7], q[8], q[9], q[10], q[11], (int)q[12], (int)q[13]};
        run_env<AcrobotD>(p, n, steps, rng, actions, random_policy, state_io, (double*)reward_out, terminal_out, t_io, action_out, do_reset_first);
        return 0;
    }
    return -1;
}
}
