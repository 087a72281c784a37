"""The kernels' device source, compiled for the host, against the oracle (no GPU).

csrc/jl_device.cuh (Julia sin / cos / mod kernels, Xoshiro256++ samplers), csrc/env_device.cuh (reset! / _step! of every env kind)
and csrc/perm.cuh (minibatch permutation) are plain C++ once the CUDA qualifiers are defined away (tests/hostdev/cuda_runtime.h);
g++ -ffp-contract=off keeps the rounding points of the nvcc -fmad=false build.  Bit-exact agreement here means an edit of the device
math is caught by the CPU suite; the `-m gpu` tests then only have to pin the kernels' plumbing."""
import ctypes as C
import itertools
import os
import subprocess

import numpy as np
import pytest

import oracle_lib as O

HERE = os.path.dirname(os.path.abspath(__file__))
HD = os.path.join(HERE, "hostdev")
CSRC = os.path.join(os.path.dirname(HERE), "reinforcementlearning.jl_b200", "csrc")
SO = os.path.join(HD, "libhostdev.so")


@pytest.fixture(scope="module")
def hd():
    srcs = [os.path.join(HD, "hostdev.cpp"), os.path.join(HD, "cuda_runtime.h")] + [os.path.join(CSRC, f) for f in ("jl_device.cuh", "env_device.cuh", "perm.cuh", "tc_split.h", "opt_path.h")]
    if not os.path.exists(SO) or any(os.path.getmtime(s) > os.path.getmtime(SO) for s in srcs):
        cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
        subprocess.check_call([cxx, "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-mfma", "-Wno-unknown-pragmas",
                               "-I", HD, "-I", CSRC, "-shared", "-o", SO, srcs[0]])
    L = C.CDLL(SO)
    vp, i32, i64, u64, f32, f64 = C.c_void_p, C.c_int, C.c_int64, C.c_uint64, C.c_float, C.c_double
    for name, res, args in (("hd_sin32", f32, [f32]), ("hd_cos32", f32, [f32]), ("hd_sin64", f64, [f64]), ("hd_cos64", f64, [f64]),
                            ("hd_mod64", f64, [f64, f64]), ("hd_perm_index", C.c_uint32, [C.c_uint32] * 3), ("hd_tc_actor_ctas", i32, [i32, i32, i64]),
                            ("hd_opt_path", i32, [i32] * 5 + [i64] + [i32] * 5), ("hd_rand_oneto", i64, [vp, u64]),
                            ("hd_env_run", i32, [i32, vp, i64, i32, vp, vp, i32, vp, vp, vp, vp, vp, i32])):
        fn = getattr(L, name)
        fn.restype, fn.argtypes = res, args
    return L


def test_julia_math_kernels_bitwise(hd):
    o = O.lib()
    rng = np.random.default_rng(0)
    xs32 = np.concatenate([rng.uniform(-0.3, 0.3, 4000), rng.uniform(-30, 30, 4000), rng.standard_normal(2000) * 1e-4,
                           [0.0, -0.0, 0.78539816, 0.7853982, 1e-5, 2.4414062e-4, 3.4526698e-4, 100.0, -1000.5]]).astype(np.float32)
    for x in xs32:
        assert hd.hd_sin32(x) == o.orc_sin32(x) or (np.isnan(hd.hd_sin32(x)) and np.isnan(o.orc_sin32(x))), x
        assert hd.hd_cos32(x) == o.orc_cos32(x), x
    xs64 = np.concatenate([rng.uniform(-0.3, 0.3, 4000), rng.uniform(-1e3, 1e3, 4000), rng.uniform(-7.2, 7.2, 6000), rng.standard_normal(1000) * 1e-9,
                           np.pi / 2 * np.arange(-6, 7) + 1e-9, np.pi / 2 * np.arange(-6, 7), [0.0, 0.7853981633974483, 1e6 + 0.1]])
    for x in xs64:
        assert hd.hd_sin64(x) == o.orc_sin64(x), x
        assert hd.hd_cos64(x) == o.orc_cos64(x), x
    for x, y in zip(rng.uniform(-50, 50, 3000), np.full(3000, 2 * np.pi)):
        assert hd.hd_mod64(x, y) == o.orc_mod64(x, y)
    assert np.float32(np.sin(np.float64(xs32[:8000]))).tolist() != [] and np.mean(
        [hd.hd_sin32(x) == np.float32(np.sin(np.float64(x))) for x in xs32[:8000]]) > 0.999      # sanity: these ARE sines


def test_samplers_and_permutation_bitwise(hd):
    o = O.lib()
    for n in (2, 3, 7, 4096, (1 << 63) + 12345):
        s1 = O.splitmix_states_fast(1, n & 0xFFFF)[0].copy(); s2 = s1.copy()
        for _ in range(200):
            assert hd.hd_rand_oneto(O._p(s1), n) == o.orc_rng_oneto(O._p(s2), n)
        assert np.array_equal(s1, s2)
    for n, key in ((1, 5), (2, 9), (5, 1), (1000, 77), (4096, 123), (65536 * 32, 12345), (100003, 0xFFFFFFFF)):
        qs = range(n) if n <= 5000 else list(range(0, n, max(1, n // 3000)))
        assert all(hd.hd_perm_index(q, n, key) == o.orc_perm_index(q, n, key) for q in qs)
    assert sorted(hd.hd_perm_index(q, 1000, 77) for q in range(1000)) == list(range(1000))


# (hostdev kind, oracle kind, dtype, discrete action count or None, action bounds)
CASES = [
    pytest.param(0, O.KIND_CARTPOLE, "f32", 2, None, id="CartPole-f32"),
    pytest.param(5, O.KIND_CARTPOLE, "f64", 2, None, id="CartPole-f64"),
    pytest.param(1, O.KIND_PENDULUM, "f32", None, 2.0, id="Pendulum-continuous"),
    pytest.param(6, O.KIND_PENDULUM, "f32", 3, None, id="Pendulum-discrete"),
    pytest.param(2, O.KIND_MOUNTAINCAR, "f32", 3, None, id="MountainCar"),
    pytest.param(3, O.KIND_CARTPOLE_CONT, "f32", None, 1.0, id="CartPole-continuous"),
    pytest.param(4, O.KIND_MOUNTAINCAR_CONT, "f32", None, 1.0, id="MountainCar-continuous"),
    # T = Float64: the reference constructors' default for Pendulum / MountainCar (PendulumEnv.jl:42, MountainCarEnv.jl:67)
    pytest.param(7, O.KIND_PENDULUM, "f64", None, 2.0, id="Pendulum-f64-continuous"),
    pytest.param(8, O.KIND_PENDULUM, "f64", 3, None, id="Pendulum-f64-discrete"),
    pytest.param(9, O.KIND_MOUNTAINCAR, "f64", 3, None, id="MountainCar-f64"),
    pytest.param(10, O.KIND_MOUNTAINCAR_CONT, "f64", None, 1.0, id="MountainCar-f64-continuous"),
    pytest.param(11, O.KIND_ACROBOT, "f64", 3, None, id="Acrobot-f64"),
]


def _oracle(okind, dtype, n, seeds, discrete_pendulum):
    params = None
    if discrete_pendulum:
        params = O.default_params(O.KIND_PENDULUM, dtype).copy()
        params[8] = 0
    return O.OracleVecEnv(okind, n, seeds, dtype=dtype, params=params)


@pytest.mark.parametrize("hkind,okind,dtype,n_act,bound", CASES)
def test_env_step_and_auto_reset_bitwise(hd, hkind, okind, dtype, n_act, bound):
    n, steps = 1200, 260                                   # 260 > max_steps = 200: the time limit resets every env at least once
    seeds = O.splitmix_states_fast(n, 31 + hkind)
    ref = _oracle(okind, dtype, n, seeds, hkind in (6, 8))
    ref.reset(force=True)
    T = np.float64 if dtype == "f64" else np.float32
    state = np.ascontiguousarray(ref.get(O.F_STATE))       # (n, NS): one env's state contiguous = the device layout
    rng = ref.get(O.F_RNG).copy()
    t = ref.get(O.F_T).copy()
    r = np.random.default_rng(hkind)
    if n_act:
        A = r.integers(1, n_act + 1, (n, steps)).astype(np.int32)
    else:
        A = r.uniform(-bound, bound, (n, steps)).astype(T)          # a continuous action is a T
    A = np.asfortranarray(A)
    rew = np.zeros((n, steps), T, order="F"); term = np.zeros((n, steps), np.uint8, order="F")
    assert hd.hd_env_run(hkind, O._p(ref.params), n, steps, O._p(rng), O._p(A), 0, O._p(state), O._p(rew), O._p(term), O._p(t), None, 0) == 0
    for k in range(steps):
        assert ref.step(A[:, k], auto_reset=True) == 0
        assert np.array_equal(ref.get(O.F_REWARD).view(np.uint8), np.ascontiguousarray(rew[:, k]).view(np.uint8)), k
        assert np.array_equal(ref.get(O.F_TERMINAL) & 1, term[:, k]), k
    assert term.sum() >= n                                  # every env finished at least one episode
    assert np.array_equal(ref.get(O.F_STATE).view(np.uint8), state.view(np.uint8))
    assert np.array_equal(ref.get(O.F_RNG), rng) and np.array_equal(ref.get(O.F_T), t)


@pytest.mark.parametrize("hkind,okind,dtype,n_act,bound", [c for c in CASES if c.values[3]])
def test_env_reset_and_random_policy_bitwise(hd, hkind, okind, dtype, n_act, bound):
    n, steps = 800, 230
    seeds = O.splitmix_states_fast(n, 77 + hkind)
    ref = _oracle(okind, dtype, n, seeds, hkind in (6, 8))  # the constructor resets once (CartPoleEnv.jl:77) ...
    ref.reset(force=True)                                   # ... and run() resets again before the first step (run.jl:46)
    T = np.float64 if dtype == "f64" else np.float32
    ns = O.NS[okind]
    state = np.zeros((n, ns), T); rng = seeds.copy(); t = np.full(n, 99, np.int32)
    dummy_r = np.zeros((n, 1), T); dummy_t = np.zeros((n, 1), np.uint8)
    for _ in range(2):                                      # two reset!() calls on the raw streams, no steps
        assert hd.hd_env_run(hkind, O._p(ref.params), n, 0, O._p(rng), None, 0, O._p(state), O._p(dummy_r), O._p(dummy_t), O._p(t), None, 1) == 0
    assert np.array_equal(ref.get(O.F_STATE).view(np.uint8), state.view(np.uint8))
    assert np.array_equal(ref.get(O.F_RNG), rng) and not t.any()
    # RandomPolicy sharing the env's stream (random_policy.jl:18-32): draw, step, auto-reset
    rew = np.zeros((n, steps), T, order="F"); term = np.zeros((n, steps), np.uint8, order="F"); last = np.zeros(n, np.int32)
    assert hd.hd_env_run(hkind, O._p(ref.params), n, steps, O._p(rng), None, 1, O._p(state), O._p(rew), O._p(term), O._p(t), O._p(last), 0) == 0
    for k in range(steps):
        a = ref.step_random(auto_reset=True)
        assert np.array_equal(ref.get(O.F_TERMINAL) & 1, term[:, k]), k
    assert np.array_equal(a, last)
    assert np.array_equal(ref.get(O.F_STATE).view(np.uint8), state.view(np.uint8))
    assert np.array_equal(ref.get(O.F_RNG), rng) and np.array_equal(ref.get(O.F_T), t)


def _f32(v):
    return float(np.float32(v))


CUSTOM = [
    # CartPoleEnvParams{Float32}(; gravity = 9.0, masscart = 1.3, masspole = 0.2, halflength = 0.4, forcemag = 7.5, max_steps = 50, dt = 0.03,
    #                            thetathreshold = 9.0, xthreshold = 1.5): derived fields in Float64, then -> T (CartPoleEnv.jl:22-46)
    pytest.param(0, O.KIND_CARTPOLE, "f32", 2,
                 [_f32(9.0), _f32(1.3), _f32(0.2), _f32(1.3 + 0.2), _f32(0.4), _f32(0.2 * 0.4), _f32(7.5), _f32(0.03), _f32(9.0 * np.pi / 180), _f32(1.5), 50],
                 id="CartPole-f32-custom"),
    pytest.param(5, O.KIND_CARTPOLE, "f64", 2, [9.0, 1.3, 0.2, 1.3 + 0.2, 0.4, 0.2 * 0.4, 7.5, 0.03, 9.0 * np.pi / 180, 1.5, 50], id="CartPole-f64-custom"),
    # PendulumEnv(; T = Float32, max_speed = 6, max_torque = 1.5, g = 9.81, m = 0.8, l = 1.2, dt = 0.02, max_steps = 77, continuous = false, n_actions = 5)
    pytest.param(6, O.KIND_PENDULUM, "f32", 5, [6.0, 1.5, _f32(9.81), _f32(0.8), _f32(1.2), _f32(0.02), 77, 5, 0], id="Pendulum-discrete5-custom"),
    # MountainCarEnv(; T = Float32, max_speed = 0.05, goal_pos = 0.3, power = 0.002, gravity = 0.003, max_steps = 120)
    pytest.param(2, O.KIND_MOUNTAINCAR, "f32", 3, [_f32(-1.2), _f32(0.6), _f32(0.05), _f32(0.3), 0.0, _f32(0.002), _f32(0.003), 120], id="MountainCar-custom"),
]


@pytest.mark.parametrize("hkind,okind,dtype,n_act,params", CUSTOM)
def test_env_with_non_default_parameters_bitwise(hd, hkind, okind, dtype, n_act, params):
    """a1: every field of the params structs reaches the arithmetic (nothing is a baked-in default)."""
    n, steps = 600, 160
    seeds = O.splitmix_states_fast(n, 500 + hkind)
    q = np.array(params, np.float64)
    ref = O.OracleVecEnv(okind, n, seeds, dtype=dtype, params=q)
    ref.reset(force=True)
    T = np.float64 if dtype == "f64" else np.float32
    state = np.ascontiguousarray(ref.get(O.F_STATE)); rng = ref.get(O.F_RNG).copy(); t = ref.get(O.F_T).copy()
    A = np.asfortranarray(np.random.default_rng(9).integers(1, n_act + 1, (n, steps)).astype(np.int32))
    rew = np.zeros((n, steps), T, order="F"); term = np.zeros((n, steps), np.uint8, order="F")
    assert hd.hd_env_run(hkind, O._p(q), n, steps, O._p(rng), O._p(A), 0, O._p(state), O._p(rew), O._p(term), O._p(t), None, 0) == 0
    for k in range(steps):
        assert ref.step(A[:, k], auto_reset=True) == 0
        assert np.array_equal(ref.get(O.F_REWARD).view(np.uint8), np.ascontiguousarray(rew[:, k]).view(np.uint8)), k
        assert np.array_equal(ref.get(O.F_TERMINAL) & 1, term[:, k]), k
    assert term.sum() >= n
    assert np.array_equal(ref.get(O.F_STATE).view(np.uint8), state.view(np.uint8))
    assert np.array_equal(ref.get(O.F_RNG), rng) and np.array_equal(ref.get(O.F_T), t)


def test_actor_critic_cta_split_rule(hd):
    """tc_split.h: the split of the 148 persistent CTAs of the loss + backward kernel.  Pinned: the two measured optima (79 : 69 for the
    4 096-tile BASELINE minibatch, 80 : 68 for the 8 192-tile Pendulum batch), the bounds the fused optimiser step relies on, and
    optimality of the returned split under the cost model for arbitrary tile counts."""
    assert hd.hd_tc_actor_ctas(148, 0, 4096) == 79 and hd.hd_tc_actor_ctas(148, 1, 8192) == 80
    import math
    for grid in (148, 132, 2, 8):
        for gaussian, r in ((0, 0.87), (1, 0.85)):
            for nt in list(range(0, 300)) + [511, 512, 1000, 4096, 8192, 65536, 10 ** 7]:
                na = hd.hd_tc_actor_ctas(grid, gaussian, nt)
                assert grid // 2 <= na <= min(grid // 2 + 8, grid - 1) or (grid == 2 and na == 1)
                cost = lambda a: max(math.ceil(nt / a), r * math.ceil(nt / (grid - a)))
                cands = [a for a in range(grid // 2, min(grid // 2 + 8, grid - 1) + 1)]
                assert cost(na) <= min(cost(a) for a in cands) + 1e-9


FUSED_TAIL, ONE_KERNEL, ONE_KERNEL_XCHG, NCCL_CHAIN = range(4)


def test_optimiser_step_path_rule(hd):
    """opt_path.h: which kernels run an optimiser step, for every combination of its inputs, including the sharded NCCL rows that no
    single-GPU test reaches.  The fused tail's size limits are pinned at the BASELINE network (9 155 parameters, 148 CTAs, <= 82
    partial rows) and just past each limit."""
    fits = dict(np=9155, grid=148, rows=82, sm=148)
    misfits = [dict(fits, np=148 * 512 + 1),            # > 512 parameters per CTA
               dict(fits, rows=83),                      # 62 x 83 staged floats > 10 x 512
               dict(fits, grid=258, sm=258),             # more CTAs than the staged loss rows allow
               dict(fits, sm=146)]                       # not co-resident
    for tail_fits, shape in [(True, fits)] + [(False, m) for m in misfits]:
        for world in (1, 2, 8):
            for p2p in ((False,) if world == 1 else (False, True)):        # a peer exchange needs peers
                for exclusive, fused, tc, inbox, cores in itertools.product((False, True), repeat=5):
                    got = hd.hd_opt_path(world, p2p, exclusive, fused, tc, shape["np"], shape["grid"], shape["rows"], shape["sm"], inbox, cores)
                    if fused and tc and tail_fits and (world == 1 or (p2p and exclusive and inbox)):
                        want = FUSED_TAIL
                    elif (world > 1 and not p2p) or not cores:
                        want = NCCL_CHAIN       # also on one GPU when the reduce + Adam grid cannot be co-resident
                    else:
                        want = ONE_KERNEL_XCHG if p2p else ONE_KERNEL   # (a gradient too large for the inbox is refused by the launcher)
                    assert got == want, (world, p2p, exclusive, fused, tc, inbox, cores, shape)
