#!/usr/bin/env python
"""bench.py — env-steps/s of the full PPO iteration on 65 536 batched CartPole envs
(BASELINE.json metric / configs[1]; configs[3] when --gpus > 1: the same 65 536 envs sharded
by index, one gradient exchange per optimiser step).

One "step" = one PPO iteration = rollout of T = 32 env steps for every env (policy inference +
env step + trajectory push fused on the device) + GAE/returns/normalisation + 4 epochs x 4
minibatches of {loss + backward, reduce, clip + Adam}  =  N*T env-steps, replayed as ONE CUDA
graph launch (b200rl_onpolicy_iterate).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference-shaped CPU arm (oracle port, all host cores)
    python bench.py --config c3|c5                           # BASELINE configs[2] (Pendulum A2C) / configs[4] (DQN 1M replay), 1 GPU
    python bench.py ... --dump-outputs DIR                   # also write what the last timed step computed, as DIR/<name>.npy

Prints ONE JSON line (see DESIGN.md "Measurement").  Timing: one CUDA event pair per step on the
launching stream (L2 flushed between steps, outside the timed region), NO host synchronisation
inside the loop (the host runs ahead; the intervals are read after the closing barrier),
barrier + synchronise around the loop, max over ranks.

Inputs are seeded, so two runs with the same arguments compute from the same inputs; --dump-outputs
lets two builds be compared output for output.  The benchmark writes nothing into the source tree."""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

sys.dont_write_bytecode = True   # no __pycache__ in the tree (it may be read-only)
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_ENVS, T_ROLLOUT, N_EPOCHS, N_MICRO, HIDDEN = 65536, 32, 4, 4, 64
# algorithmic work per sample (SURVEY §8d): MLP forward actor 8 960 + critic 8 832 FLOP; fwd+bwd = 3x
FLOP_FWD = 2 * (4 * 64 + 64 * 64 + 64 * 2) + 2 * (4 * 64 + 64 * 64 + 64 * 1)
FLOP_FWD_BWD = 3 * FLOP_FWD
BYTES_ENV_STEP = 49 + 8          # state 16R+16W, action 4R, t 4R+4W, reward 4W, flag 1W (+ episode-return 4R+4W)
BYTES_GAE = 17 + 8               # r 4, v 4, term 1 read; adv 4, ret 4 write (+ 8: returns)
BYTES_K7_SAMPLE = 32             # SURVEY §8d: s 16 + a 4 + logp_old 4 + adv 4 + ret 4 per sample per epoch (= one packed record)
BYTES_LOOP_ENV_STEP = 235        # SURVEY §8d: full PPO iteration per env-step (49 + 33 + 25 + 4 x 32)
METRIC = "env-steps/sec at 65536 CartPole envs (full PPO iteration: rollout T=32 + GAE + 4 epochs x 4 minibatches)"
PHASE_BASE = 448                 # timer slots used by the per-phase breakdown
DUMP_MAX_BYTES = 64 << 20        # --dump-outputs: cap on everything written
DUMP_ENVS = 16384                # --dump-outputs: rollout columns kept (a fixed, seeded sample when there are more envs)


def write_outputs(out_dir, arrays):
    """--dump-outputs: every array as out_dir/<name>.npy, float32 arrays as they are, anything else as float64 (exact for the
    integer actions, flags and replay keys)."""
    arrays = {k: np.ascontiguousarray(a, np.float32 if np.asarray(a).dtype == np.float32 else np.float64) for k, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise ValueError(f"--dump-outputs: {total} bytes exceed the {DUMP_MAX_BYTES}-byte cap")
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def dump_env_sample(n):
    """Env columns --dump-outputs keeps: all of them up to DUMP_ENVS, else DUMP_ENVS indices drawn with a fixed seed (sorted)."""
    if n <= DUMP_ENVS:
        return np.arange(n)
    return np.sort(np.random.default_rng(0).choice(n, DUMP_ENVS, replace=False))


def onpolicy_outputs(pkg, agent, net):
    """What one on-policy iteration hands its caller: the updated parameters, and the rollout it trained on (with values,
    advantages, returns and the advantage normalisation) for the env columns of dump_env_sample."""
    R = pkg.learners
    idx = dump_env_sample(agent.n)
    out = {"params": net.get(), "adv_norm": agent.rollout(R.ROLL_NORM), "env_index": idx}
    for name, f in (("state", R.ROLL_STATE), ("action", R.ROLL_ACTION), ("logp", R.ROLL_LOGP), ("reward", R.ROLL_REWARD),
                    ("terminal", R.ROLL_TERMINAL), ("value", R.ROLL_VALUE), ("advantage", R.ROLL_ADV), ("return", R.ROLL_RET)):
        a = agent.rollout(f)
        out[name] = a[:, idx] if f == R.ROLL_STATE else a[idx]
    return out


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops", 1590.0), "measured"
    return 6650.0, 1590.0, "fallback"


def _physical_indices(n):
    """NVML / nvidia-smi index of visible device 0..n-1 (CUDA_VISIBLE_DEVICES given as integers; identity otherwise)."""
    cvd = os.environ.get("CUDA_VISIBLE_DEVICES", "")
    try:
        ids = [int(x) for x in cvd.split(",") if x.strip() != ""]
        if len(ids) >= n:
            return ids[:n]
    except ValueError:
        pass
    return list(range(n))


class ClockSampler:
    """SM clocks / throttle reasons / power of every GPU of the job, sampled by ONE thread of rank 0 (NVML in-process —
    no nvidia-smi processes spawned next to the timed loop; falls back to a single `nvidia-smi -lms` reader if the NVML
    binding is missing).  Started before warm-up; the summary covers the window marked by begin() / end()."""
    R_SW_POWER_CAP, R_HW_SLOWDOWN, R_SW_THERMAL, R_HW_THERMAL = 0x4, 0x8, 0x20, 0x40

    def __init__(self, n_gpus, period=0.01):
        self.ids, self.period, self.rows, self.t0, self.t1 = _physical_indices(n_gpus), period, [], None, None
        self.stop_flag, self.thread, self.proc, self.kind = False, None, None, None

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            self.nv = nv
            self.handles = [nv.nvmlDeviceGetHandleByIndex(i) for i in self.ids]
            self.max_sm = [float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)) for h in self.handles]
            self.kind = "nvml"
            self.thread = threading.Thread(target=self._loop_nvml, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.kind = None
        try:
            q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
            self.proc = subprocess.Popen(["nvidia-smi", "-i", ",".join(map(str, self.ids)), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.kind = "nvidia-smi"
            self.thread = threading.Thread(target=self._loop_smi, daemon=True)
            self.thread.start()
        except Exception:
            self.kind = None

    def _loop_nvml(self):
        nv = self.nv
        reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self.stop_flag:
            now = time.perf_counter()
            for k, h in enumerate(self.handles):
                try:
                    self.rows.append((now, k, float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)), self.max_sm[k],
                                      nv.nvmlDeviceGetPowerUsage(h) / 1000.0, int(reasons(h))))
                except Exception:
                    pass
            time.sleep(self.period)

    def _loop_smi(self):
        names = [self.R_HW_SLOWDOWN, self.R_HW_THERMAL, self.R_SW_THERMAL, self.R_SW_POWER_CAP]
        for line in self.proc.stdout:
            p = [x.strip() for x in line.split(",")]
            if len(p) < 8:
                continue
            try:
                mask = sum(b for b, v in zip(names, p[4:8]) if v.lower().startswith("active"))
                self.rows.append((time.perf_counter(), self.ids.index(int(p[0])), float(p[1]), float(p[2]), float(p[3]), mask))
            except Exception:
                pass

    def begin(self):
        self.t0 = time.perf_counter()

    def end(self):
        self.t1 = time.perf_counter()

    def stop(self):
        if self.kind is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock sampler unavailable"]}
        time.sleep(2.5 * self.period)
        self.stop_flag = True
        if self.proc:
            self.proc.terminate()
        rows = [r for r in self.rows if self.t0 is not None and self.t0 <= r[0] <= (self.t1 or 1e300)]
        window = "timed region"
        if len(rows) < max(2, len(self.ids)):   # a timed region shorter than the sampling period: fall back to everything under load
            rows, window = [r for r in self.rows if r[2] > 0.6 * r[3]] or self.rows, "warm-up + timed region (timed region shorter than the sampling period)"
        sm = [r[2] for r in rows]
        mask = 0
        for r in rows:
            mask |= r[5]
        reasons = [n for b, n in ((self.R_HW_SLOWDOWN, "hw_slowdown"), (self.R_HW_THERMAL, "hw_thermal_slowdown"), (self.R_SW_THERMAL, "sw_thermal_slowdown"),
                                  (self.R_SW_POWER_CAP, "sw_power_cap")) if mask & b]
        per_gpu = {}
        for r in rows:
            per_gpu.setdefault(r[1], []).append(r[2])
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max((r[3] for r in rows), default=None), "reasons": reasons,
                "samples": len(rows), "power_w_max": max((r[4] for r in rows), default=None), "source": self.kind, "window": window,
                "sm_mhz_median_per_gpu": [float(np.median(v)) for _, v in sorted(per_gpu.items())]}


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


def usable_cores():
    """Host threads this process may really use: scheduler affinity capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(float(txt[0]) / float(txt[1]) + 0.5)))
            else:
                q = int(txt[0])
                if q > 0:
                    per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                    n = min(n, max(1, int(q / per + 0.5)))
            break
        except Exception:
            continue
    return n


def cpu_arm_setup(O, n):
    """Build the oracle-port PPO job on `n` envs and pick the OpenMP thread count that runs it fastest
    (one short calibration iteration per candidate: an over-subscribed or quota-limited box is slower
    with every hardware thread than with fewer).  The candidates come from the cores this process may use —
    NOT from OMP_NUM_THREADS, which torchrun exports as 1 for every rank.  Returns (step_fn, cores)."""
    env = O.OracleVecEnv(O.KIND_CARTPOLE, n, O.splitmix_states_fast(n, 1))
    env.reset(True)
    desc = O.ac_desc(4, HIDDEN, 2)
    p = O.glorot_params(desc, 123); m = np.zeros_like(p); v = np.zeros_like(p); bt = np.array([0.9, 0.999], np.float32)
    prng = O.splitmix_states_fast(n, 2).copy()
    hyper = O.hyper_array()
    counter = [0]

    def step(T=T_ROLLOUT):
        s, _ = O.ppo_iteration(env, desc, hyper, p, m, v, bt, prng, T, N_EPOCHS, N_MICRO, counter[0])
        counter[0] += 1
        return s

    top = max(1, usable_cores())
    cands = sorted({top, max(1, top // 2), max(1, top // 4), min(top, 32), min(top, 16), min(top, 8)}, reverse=True)
    best, best_s = top, None
    for c in cands:
        O.lib().orc_set_threads(c)
        s = min(step(T=8), step(T=8))   # best of two short iterations (8-step rollout + the full update shape) per candidate
        if best_s is None or s < best_s:
            best, best_s = c, s
    O.lib().orc_set_threads(best)
    return step, best


def run_reference(args):
    """The reference's own CPU implementation of the path cannot run here (Julia absent, RLZoo /
    MultiThreadEnv not in the snapshot): this arm times the oracle port — per-env heap objects,
    OpenMP parallel-for over envs (Threads.@threads stand-in), Appendix-B PPO update — on all host
    cores, each step a bounded sample (8192 of the 65 536 envs)."""
    rank, _, world = dist_env()
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    n = args.cpu_envs
    step, cores = cpu_arm_setup(O, n)
    for w in range(args.warmup):
        step()
    secs = [step() for _ in range(args.steps)]
    total = float(np.sum(secs))
    value = n * T_ROLLOUT * args.steps / total
    sample = f"{n} of {N_ENVS} envs per step (same T, epochs, minibatches)"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "env-steps/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000.0 * total / args.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "PPO 2x64 actor-critic on batched CartPoleEnv{Float32}, T=32, 4 epochs x 4 minibatches", "n_envs": n,
                   "parallelism": f"cpu{cores}", "note": "oracle port of the reference path; bounded sample; OpenMP threads chosen from the usable host cores "
                                                          f"({usable_cores()}), independent of OMP_NUM_THREADS"},
        "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


class Job:
    """ctx + communicator plumbing shared by the configs (one process per GPU; torch.distributed only ships the NCCL id and
    the 64-byte IPC handles, and provides the closing barrier / max-over-ranks)."""

    def __init__(self, args):
        self.rank, self.local_rank, self.world = dist_env()
        if self.world != args.gpus and self.world > 1:
            args.gpus = self.world
        import __graft_entry__ as g
        self.pkg = pkg = g.load_package()
        self.dist = None
        if self.world > 1:
            import torch
            import torch.distributed as dist
            torch.cuda.set_device(self.local_rank)
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
            self.dist = dist
        self.ctx = ctx = pkg.Context(self.local_rank)
        self.peer_exchange = False
        if self.world > 1:
            import ctypes as C
            import torch
            idbuf = torch.zeros(128, dtype=torch.uint8, device="cuda")
            if self.rank == 0:
                raw = (C.c_char * 128)()
                pkg._lib.check(ctx.lib.b200rl_comm_unique_id(raw))
                idbuf.copy_(torch.frombuffer(bytearray(raw.raw), dtype=torch.uint8))
            self.dist.broadcast(idbuf, 0)
            raw = bytes(idbuf.cpu().numpy().tobytes())
            pkg._lib.check(ctx.lib.b200rl_comm_init(ctx.h, self.world, self.rank, raw))
            if os.environ.get("B200RL_P2P", "1") != "0":
                from b200rl import sharding as _sh
                self.peer_exchange = _sh.attach_peer_exchange(ctx, self.rank, self.world, self.all_gather_bytes)

    def all_gather_bytes(self, b):
        import torch
        t = torch.frombuffer(bytearray(b), dtype=torch.uint8).cuda()
        out = [torch.empty_like(t) for _ in range(self.world)]
        self.dist.all_gather(out, t)
        return [bytes(o.cpu().numpy().tobytes()) for o in out]

    def barrier(self):
        self.ctx.sync()
        if self.dist is not None:
            import torch
            self.dist.barrier(device_ids=[self.local_rank])
            torch.cuda.synchronize()

    def max_over_ranks(self, x):
        if self.dist is None:
            return float(x)
        import torch
        tt = torch.tensor([x], dtype=torch.float64, device="cuda")
        self.dist.all_reduce(tt, op=self.dist.ReduceOp.MAX)
        return float(tt.item())

    def gather_objects(self, obj):
        if self.dist is None:
            return [obj]
        out = [None] * self.world
        self.dist.all_gather_object(out, obj)
        return out

    def close(self):
        if self.dist is not None:
            self.dist.destroy_process_group()
        self.ctx.close()


def timed_steps(job, step_fn, steps, sampler=None):
    """K steps, one event pair each, L2 flushed between them outside the timed region, no host sync inside the loop.
    Returns the max over ranks of the summed device time (ms)."""
    ctx = job.ctx
    total_ms, done = 0.0, 0
    job.barrier()
    if sampler:
        sampler.begin()
    while done < steps:
        chunk = min(steps - done, 200)          # 2 slots per step, 400 of the 512 slots
        for i in range(chunk):
            ctx.flush_l2()
            ctx.timer_record(2 * i)
            step_fn()
            ctx.timer_record(2 * i + 1)
        ctx.sync()
        total_ms += sum(ctx.timer_elapsed_ms(2 * i, 2 * i + 1) for i in range(chunk))
        done += chunk
    job.barrier()
    if sampler:
        sampler.end()
    return job.max_over_ranks(total_ms)


def phase_breakdown(job, agent, T, rows, reps=3):
    """Per-phase device times of one iteration on THIS rank (eager launches with events between the phases; measurement aid,
    outside the timed region): rollout | bootstrap + GAE + normalisation + record packing | sum of the loss+backward launches |
    sum of the optimiser steps (incl. the peer exchange wait on a sharded run)."""
    ctx = job.ctx
    if rows > 64:
        return None
    acc = np.zeros(4)
    ctx.phase_slots(PHASE_BASE + 1)
    try:
        for _ in range(reps):
            job.barrier()
            ctx.timer_record(PHASE_BASE)
            agent.collect(T)
            agent.update()
            ctx.sync()
            b = PHASE_BASE + 1
            acc[0] += ctx.timer_elapsed_ms(PHASE_BASE, b)
            acc[1] += ctx.timer_elapsed_ms(b, b + 1)
            for r in range(rows):
                acc[2] += ctx.timer_elapsed_ms(b + 1 + 2 * r, b + 2 + 2 * r)
                acc[3] += ctx.timer_elapsed_ms(b + 2 + 2 * r, b + 3 + 2 * r)
    finally:
        ctx.phase_slots(-1)
    acc /= reps
    return {"rank": job.rank, "rollout_ms": acc[0], "gae_norm_pack_ms": acc[1], "loss_backward_ms": acc[2], "optimiser_exchange_ms": acc[3],
            "sum_ms": float(acc.sum())}


def run_c2(args):
    job = Job(args)
    pkg, ctx, rank, world = job.pkg, job.ctx, job.rank, job.world
    from b200rl import sharding
    T = T_ROLLOUT
    cfg = pkg.onpolicy_config(update_freq=T, n_epochs=N_EPOCHS, n_microbatches=N_MICRO)
    rows = N_EPOCHS * N_MICRO
    glorot = lambda seed: sharding.glorot_actor_critic(seed, 4, HIDDEN, 2)

    def make(n_total, host_actions):
        lo, hi = sharding.shard_range(n_total, rank, world)
        states = lambda seed: sharding.splitmix_states(seed, lo, hi)      # streams keyed by GLOBAL env index
        env = pkg.B200VecEnv(ctx, "CartPole", hi - lo, states(0x9E3779B97F4A7C15), auto_reset=True)
        net = pkg.Network(ctx, 4, HIDDEN, 2, glorot(123))
        agent = pkg.OnPolicyAgent(ctx, net, env, cfg, states(0x1234567), host_actions=host_actions)
        env.reset_(is_force=True)
        return env, net, agent

    sampler = None
    if rank == 0:
        sampler = ClockSampler(world)
        sampler.start()            # ONE sampler for the whole job, before warm-up
    n_total = args.envs
    n = n_total // world
    env, net, agent = make(n_total, False)
    ctx.flush_l2()                 # allocates the flush buffer here, not inside the timed loop
    for _ in range(max(args.warmup, 2)):   # >= 2: the first iteration runs eagerly, the second captures the graph
        agent.iterate(1)
    launches0 = ctx.launch_count()
    total_ms = timed_steps(job, lambda: agent.iterate(1), args.steps, sampler)
    launches = ctx.launch_count() - launches0
    if args.dump_outputs and rank == 0:   # parameters are replicated; the rollout is rank 0's shard
        write_outputs(args.dump_outputs, onpolicy_outputs(pkg, agent, net))
    clk = sampler.stop() if sampler else None
    graph = agent.graph_active()
    value = n_total * T * args.steps / (total_ms / 1000.0)
    stats = env.episode_stats()

    phases = job.gather_objects(phase_breakdown(job, agent, T, rows))
    # replicas of a sharded run must stay bit-identical (every rank adds the exchanged gradients in rank order): compare a checksum
    pbits = np.frombuffer(net.get().tobytes(), dtype=np.uint32)
    chks = job.gather_objects((int(pbits.astype(np.uint64).sum()), int(np.bitwise_xor.reduce(pbits))))
    replicas_identical = (len(set(chks)) == 1) if chks else None

    # ---- weak-scaling line (N > 1): 65 536 envs PER GPU, same iteration ---------------------------------
    weak = None
    if world > 1 and not args.no_weak:
        env_w, net_w, agent_w = make(N_ENVS * world, False)
        for _ in range(max(args.warmup, 2)):
            agent_w.iterate(1)
        k_w = max(3, min(args.steps, 10))
        ms_w = timed_steps(job, lambda: agent_w.iterate(1), k_w)
        weak = {"envs_per_gpu": N_ENVS, "n_envs": N_ENVS * world, "steps": k_w, "ms_per_step": ms_w / k_w,
                "value": N_ENVS * world * T * k_w / (ms_w / 1000.0), "unit": "env-steps/s", "scaling": "weak"}
        agent_w.close(); net_w.close(); env_w.close()

    # ---- e2e: the reference-facing stage protocol with HOST action buffers every step ---------
    e2e = None
    if not args.no_e2e:
        env2, net2, agent2 = make(n_total, True)
        agent2.fetch_stats = True
        k_e2e = max(1, min(args.steps, 5))
        pkg.run(agent2, env2, pkg.StopAfterNSteps(T * max(1, min(args.warmup, 2))), pkg.DeviceEpisodeStats())
        job.barrier()
        t0 = time.perf_counter()
        pkg.run(agent2, env2, pkg.StopAfterNSteps(T * k_e2e), pkg.DeviceEpisodeStats())
        ctx.sync()
        sec = job.max_over_ranks(time.perf_counter() - t0)
        e2e = {"value": n_total * T * k_e2e / sec, "unit": "env-steps/s", "h2d_bytes_per_step": int(T * n * 4),
               "d2h_bytes_per_step": int(T * n * 4 + N_EPOCHS * N_MICRO * 6 * 4 + 32), "steps": k_e2e,
               "note": "run(agent, env, StopAfterNSteps, hook): plan! returns host actions, act! takes host actions, per-update loss read-back"}
        agent2.close(); net2.close(); env2.close()

    # ---- roofline of the dominant kernel + per-kernel times (CUDA events, back-to-back launches) ----
    hbm_peak, tf_peak, peak_kind = measured_peaks()
    B_local = n * T // N_MICRO
    k_loss = agent.time_kernel(0, 10)
    k_act = agent.time_kernel(1, 20)
    tc_on = os.environ.get("B200RL_TC", "1") != "0"
    k_loss_ffma = k_act_ffma = None
    if tc_on:   # the FP32 CUDA-core variants of the same kernels, for the record
        pkg._lib.check(ctx.lib.b200rl_set_tensor_cores(0))
        k_loss_ffma = agent.time_kernel(0, 10)
        k_act_ffma = agent.time_kernel(1, 20)
        pkg._lib.check(ctx.lib.b200rl_set_tensor_cores(1))
    k_gae = agent.time_kernel(3, 20)
    k_adam = agent.time_kernel(4, 20)
    k_env = agent.time_kernel(2, 20)
    ach_tf = B_local * FLOP_FWD_BWD / (k_loss * 1e-3) / 1e12
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        try:
            tj = json.load(open(tpath))
            traffic = tj.get("ac_loss_grad_tc_kernel" if tc_on else "ac_loss_grad_kernel", tj.get("ac_loss_grad_kernel"))
        except Exception:
            traffic = None
    ms_step = total_ms / args.steps
    share = (N_EPOCHS * N_MICRO * k_loss) / ms_step
    kname = ("ac_loss_grad_tc_kernel (PPO loss + backward, one minibatch; 64x64 GEMMs on tcgen05 kind::f16 as a 3-term fp16 split "
             "hi*hi + hi*lo + lo*hi, FP32 accumulate in TMEM; the optimiser step runs in the tail of the same launch)"
             if tc_on else "ac_loss_grad_kernel<64> (PPO loss + backward, one minibatch; FP32 FFMA)")
    roofline = {"kernel": kname, "bound": "tensor", "achieved": ach_tf, "peak": tf_peak,
                "unit": "TFLOP/s", "frac": ach_tf / tf_peak, "traffic": traffic, "peak_kind": f"bf16 dense GEMM burst, {peak_kind}",
                "executed_tensor": {"tflops": 3.0 * ach_tf, "peak": tf_peak, "frac": 3.0 * ach_tf / tf_peak,
                                    "note": "the 1e-5 parity bar needs ~22 mantissa bits: every algorithmic product is three kind::f16 tensor-core products "
                                            "(fp16 hi/lo split, K = 16 per instruction); executed tensor work / the measured 16-bit dense peak"},
                "algorithmic_bytes_per_launch": B_local * BYTES_K7_SAMPLE,
                "note": "achieved = algorithmic FP32 FLOPs (53,376 per sample) / event time; as a fraction of the FP32 CUDA-core peak (~72 TFLOP/s @1.9 GHz) = %.3f"
                        % (ach_tf / 72.0),
                "ms_per_launch": k_loss, "ms_per_launch_fp32_ffma_variant": k_loss_ffma, "share_of_step": share,
                "ms_per_launch_note": "loss + backward alone (the timed iteration additionally runs reduce + clip + Adam in the tail of each launch)",
                "whole_loop_hbm": {"gbs": value * BYTES_LOOP_ENV_STEP / 1e9, "peak": hbm_peak * world, "frac": value * BYTES_LOOP_ENV_STEP / 1e9 / (hbm_peak * world),
                                   "note": "north-star figure: env-steps/s x 235 algorithmic B per env-step of the full PPO iteration (SURVEY §8d) / measured HBM "
                                           "copy bandwidth x n_gpus; the loop is issue/latency-bound, not HBM-bound"},
                "other_kernels": {
                    "policy_act_ms": k_act, "policy_act_ms_fp32_ffma_variant": k_act_ffma, "policy_act_tflops": n * FLOP_FWD / (k_act * 1e-3) / 1e12,
                    "env_step_ms": k_env, "env_step_gbs": n * BYTES_ENV_STEP / (k_env * 1e-3) / 1e9, "env_step_frac_hbm": n * BYTES_ENV_STEP / (k_env * 1e-3) / 1e9 / hbm_peak,
                    "gae_ms": k_gae, "gae_gbs_l2_resident": n * T * BYTES_GAE / (k_gae * 1e-3) / 1e9,
                    "gae_note": "at this size the 52 MB working set of the GAE kernel is L2-resident when timed back to back (ncu: 19 MB DRAM read, 0 written): "
                                "an L2 figure, not an HBM fraction; the HBM-bound sweep (4 M series) reaches 0.60 of the measured copy bandwidth (profiles/)",
                    "reduce_clip_adam_ms": k_adam,
                    "reduce_clip_adam_note": "the stand-alone optimiser-step kernel (FFMA path, ranks sharing a device, B200RL_FUSED_STEP=0); "
                                             "the tensor-core K7 runs the step in its own tail"}}

    # ---- CPU baseline (rank 0, N = 1 only): oracle port, bounded sample ------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_lib as O
        nc = args.cpu_envs
        step, cores = cpu_arm_setup(O, nc)
        s0 = step()
        reps = int(max(2, min(20, 12.0 / max(s0, 1e-3))))
        secs = [step() for _ in range(reps)]
        cpu = {"value": nc * T * reps / float(np.sum(secs)), "unit": "env-steps/s", "cores": cores, "kind": "port",
               "sample": f"{reps} PPO iterations on {nc} of {N_ENVS} envs (same T / epochs / minibatches), OpenMP over per-env heap objects, thread count picked by calibration"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": "BASELINE configs[1]: 65536 batched CartPoleEnv{Float32} + PPO (2x64 MLP actor-critic, fp32), T=32, 4 epochs x 4 minibatches, advantage normalisation",
                       "n_envs": n_total, "envs_per_gpu": n, "global_batch": n_total * T // N_MICRO, "parallelism": f"dp{world}",
                       "grad_allreduce": ("fused NVLink peer exchange inside the tail of the loss+backward kernel (reduce -> exchange -> clip -> Adam in the same launch)" if job.peer_exchange else "NCCL") if world > 1 else "none",
                       "launch": "one CUDA graph launch per iteration (b200rl_onpolicy_iterate)" if graph else "eager launches",
                       "l2": "flushed (256 MB write) between timed steps, outside the timed region",
                       "timing": "one CUDA event pair per step, no host sync inside the loop, max over ranks of the summed device time",
                       "episodes_finished_rank0": stats["episodes"]},
            "clocks": clk, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu,
            "phases_per_rank": phases, "weak_scaling": weak, "replicas_bit_identical": replicas_identical,
        }
        print(json.dumps(line), flush=True)
    agent.close(); net.close(); env.close()
    job.close()


def _dense(r, o, i):
    lim = np.sqrt(6.0 / (i + o))
    return [r.uniform(-lim, lim, (o, i)).astype(np.float32).ravel(order="F"), np.zeros(o, np.float32)]


def run_c3(args):
    """BASELINE configs[2]: 32768 batched PendulumEnv{Float32} + A2C with GAE(lambda = 0.95), continuous action (Gaussian head,
    sigma = softplus head), tanh trunks, T = 32, one epoch x one minibatch per iteration.  1 GPU."""
    job = Job(args)
    pkg, ctx = job.pkg, job.ctx
    from b200rl import sharding as sh
    n, T = 32768, 32
    r = np.random.default_rng(5)
    params = np.concatenate(_dense(r, 64, 3) + _dense(r, 64, 64) + _dense(r, 1, 64) + _dense(r, 1, 64) + _dense(r, 64, 3) + _dense(r, 64, 64) + _dense(r, 1, 64))
    cfg = pkg.onpolicy_config(update_freq=T, n_epochs=1, n_microbatches=1, algo="a2c", w_entropy=0.01, lambda_=0.95)

    def make(host_actions):
        env = pkg.B200VecEnv(ctx, "Pendulum", n, sh.splitmix_states(3, 0, n), auto_reset=True)
        net = pkg.Network(ctx, 3, 64, 1, params.copy(), act=pkg.ACT_TANH, kind=pkg.KIND_GAUSSIAN)
        agent = pkg.OnPolicyAgent(ctx, net, env, cfg, sh.splitmix_states(4, 0, n), host_actions=host_actions)
        env.reset_(True)
        return env, net, agent

    sampler = ClockSampler(1)
    sampler.start()
    env, net, agent = make(False)
    ctx.flush_l2()
    for _ in range(max(args.warmup, 2)):
        agent.iterate(1)
    l0 = ctx.launch_count()
    total_ms = timed_steps(job, lambda: agent.iterate(1), args.steps, sampler)
    launches = ctx.launch_count() - l0
    if args.dump_outputs:
        write_outputs(args.dump_outputs, onpolicy_outputs(pkg, agent, net))
    clk = sampler.stop()
    value = n * T * args.steps / (total_ms / 1000.0)
    ph = phase_breakdown(job, agent, T, 1)
    e2e = None
    if not args.no_e2e:
        env2, net2, agent2 = make(True)
        agent2.fetch_stats = True
        k = max(1, min(args.steps, 5))
        pkg.run(agent2, env2, pkg.StopAfterNSteps(T * 2), pkg.DeviceEpisodeStats())
        ctx.sync()
        t0 = time.perf_counter()
        pkg.run(agent2, env2, pkg.StopAfterNSteps(T * k), pkg.DeviceEpisodeStats())
        ctx.sync()
        sec = time.perf_counter() - t0
        e2e = {"value": n * T * k / sec, "unit": "env-steps/s", "h2d_bytes_per_step": int(T * n * 4), "d2h_bytes_per_step": int(T * n * 4 + 6 * 4 + 32),
               "steps": k, "note": "run(agent, env, StopAfterNSteps, hook) with host Float32 action buffers every step"}
        agent2.close(); net2.close(); env2.close()
    hbm_peak, tf_peak, peak_kind = measured_peaks()
    k_loss = agent.time_kernel(0, 10)
    flop = 3 * (2 * (3 * 64 + 64 * 64 + 64 * 2) + 2 * (3 * 64 + 64 * 64 + 64))
    ach = n * T * flop / (k_loss * 1e-3) / 1e12
    line = {"metric": "env-steps/sec at 32768 Pendulum envs (full A2C-GAE iteration: rollout T=32 + GAE + 1 optimiser step)", "value": value, "unit": "env-steps/s",
            "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "BASELINE configs[2]: 32768 batched PendulumEnv{Float32} + A2C with GAE(lambda=0.95), continuous action (Gaussian head), tanh 2x64 trunks, T=32",
                       "n_envs": n, "parallelism": "dp1", "l2": "flushed between timed steps, outside the timed region",
                       "launch": "one CUDA graph launch per iteration" if agent.graph_active() else "eager launches"},
            "clocks": clk, "e2e": e2e, "gpu_launches": int(launches), "phases_per_rank": [ph],
            "roofline": {"kernel": "ac_loss_grad_tc_kernel (A2C loss + backward over the whole rollout, Gaussian head, tanh; 3-term fp16 split on tcgen05 kind::f16)", "bound": "tensor",
                         "achieved": ach, "peak": tf_peak, "unit": "TFLOP/s", "frac": ach / tf_peak, "traffic": None, "peak_kind": f"bf16 dense GEMM burst, {peak_kind}",
                         "ms_per_launch": k_loss, "share_of_step": k_loss / (total_ms / args.steps)},
            "cpu_baseline": None}
    print(json.dumps(line), flush=True)
    agent.close(); net.close(); env.close()
    job.close()


def run_c5(args):
    """BASELINE configs[4]: DQN on CartPole, 1M-transition prioritised CircularArraySARTSTraces (4096 lanes x 256 frames),
    batch 4096 sample + update (4-128-128-2 Q-network, target sync every 100 updates).  One step = one optimise! call:
    prioritised sample + gather, TD loss + backward, clip + Adam, priority write-back.  1 GPU."""
    job = Job(args)
    pkg, ctx = job.pkg, job.ctx
    from b200rl import sharding as sh
    lanes, cap, B = 4096, 256, 4096
    env = pkg.B200VecEnv(ctx, "CartPole", lanes, sh.splitmix_states(7, 0, lanes), auto_reset=True)
    tr = pkg.Trajectory(ctx, 4, cap, lanes=lanes, batch_size=B, sampler_rng=sh.splitmix_states(8, 0, B), prioritized=True, default_priority=1.0)
    env.reset_(True); tr.push_env(env, first_state_only=True)
    for _ in range(cap):
        env.act_random_(); tr.push_env(env)
    r = np.random.default_rng(9)
    qparams = np.concatenate(_dense(r, 128, 4) + _dense(r, 128, 128) + _dense(r, 2, 128))
    qnet = pkg.Network(ctx, 4, 128, 2, qparams, kind=pkg.KIND_Q)
    learner = pkg.DQNLearner(ctx, qnet, tr, pkg.dqn_config(target_update_freq=100))
    sampler = ClockSampler(1)
    sampler.start()
    per_step = 50                         # one bench "step" = 50 optimise! calls (a single call is ~0.1 ms: below the event resolution we want)
    ctx.flush_l2()
    for _ in range(max(args.warmup, 3)):
        for _ in range(per_step):
            learner.update()
    l0 = ctx.launch_count()

    def step():
        for _ in range(per_step):
            learner.update()
    total_ms = timed_steps(job, step, args.steps, sampler)
    launches = ctx.launch_count() - l0
    if args.dump_outputs:   # the last optimise! call: updated Q-network, the batch it sampled, its TD errors
        out = {"params": qnet.get(), "td": learner.last_td(), "total_priority": np.array([tr.total_priority()])}
        out.update(("batch_" + k, a) for k, a in tr.batch().items())
        write_outputs(args.dump_outputs, out)
    clk = sampler.stop()
    ups = per_step * args.steps / (total_ms / 1000.0)
    # e2e: the user-facing call with the per-update statistics read back to the host (loss, grad norm, mean |td|: a D2H copy + sync per update)
    k = 100
    for _ in range(10):
        learner.update(want_stats=True)
    ctx.sync()
    t0 = time.perf_counter()
    for _ in range(k):
        learner.update(want_stats=True)
    ctx.sync()
    sec = time.perf_counter() - t0
    ms_sample = 0.0
    ctx.sync(); ctx.timer_record(0)
    for _ in range(200):
        tr.sample(fetch=False)
    ctx.timer_record(1); ctx.sync()
    ms_sample = ctx.timer_elapsed_ms(0, 1) / 200
    hbm_peak, tf_peak, peak_kind = measured_peaks()
    ms_update = total_ms / (per_step * args.steps)
    flop = 3 * 2 * (4 * 128 + 128 * 128 + 128 * 2) + 2 * 2 * (4 * 128 + 128 * 128 + 128 * 2)   # online fwd+bwd + target forward (+ none for double DQN off)
    ach = B * flop / (ms_update * 1e-3) / 1e12
    line = {"metric": "DQN updates/sec (1M-transition prioritised replay, batch 4096 sample + update)", "value": ups, "unit": "updates/s", "n_gpus": 1,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "BASELINE configs[4]: DQN on CartPole, 1,048,576-transition prioritised replay (4096 lanes x 256 frames), batch 4096, Q-net 4-128-128-2, "
                                   "target sync every 100 updates", "updates_per_bench_step": per_step, "samples_per_s": ups * B, "parallelism": "dp1",
                       "l2": "flushed between timed steps, outside the timed region"},
            "clocks": clk, "gpu_launches": int(launches),
            "e2e": {"value": k / sec, "unit": "updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": int(16 + 4 + B * 4), "steps": k,
                    "note": "learner.update(want_stats=True): loss, grad norm and the batch's TD errors read back to the host after every update"},
            "roofline": {"kernel": "whole optimise! call (sample+gather, target forward, TD loss+backward, reduce, clip+Adam, priority write-back)", "bound": "tensor",
                         "achieved": ach, "peak": tf_peak, "unit": "TFLOP/s", "frac": ach / tf_peak, "traffic": None, "peak_kind": f"bf16 dense GEMM burst, {peak_kind}",
                         "ms_per_update": ms_update, "sample_gather_ms": ms_sample, "sample_gather_gbs_at_326B": B * 326 / ms_sample / 1e6,
                         "sample_gather_frac_hbm": B * 326 / ms_sample / 1e6 / hbm_peak,
                         "note": "latency-bound at batch 4096: 5 dependent launches of a few microseconds each; the gather moves 1.3 MB"},
            "cpu_baseline": None}
    print(json.dumps(line), flush=True)
    qnet.close(); tr.close(); env.close()
    job.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="own", choices=["own", "reference"])
    ap.add_argument("--config", default="c2", choices=["c2", "c3", "c5"])
    ap.add_argument("--envs", type=int, default=N_ENVS)
    ap.add_argument("--cpu-envs", type=int, default=8192)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-weak", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy (float32 / float64, <= 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the CUDA path (--impl own)")
    if args.impl == "reference":
        run_reference(args)
    elif args.config == "c3":
        run_c3(args)
    elif args.config == "c5":
        run_c5(args)
    else:
        run_c2(args)


if __name__ == "__main__":
    main()
