#!/usr/bin/env python
"""bench.py -- env-steps/s of the Skillshot hot path on B200 (driver contract).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): physics-only, 65,536 SkillshotGame envs per
GPU, U(-1.2,1.2) float32 random actions, random starts, terminal +1/-1/0 reward,
2,000-tick limit with auto-reset.  One bench "step" = TICKS ticks of all envs
(TICKS * 65,536 env-steps per GPU), played by ss_env_step in launches of
TICKS_PER_LAUNCH fused ticks.  The action stream of a step ([TICKS, E, 2, 2]
float32 = 2.1 GB) is larger than the 126 MB L2, so every timed iteration streams
it from HBM ("inputs larger than L2"); the 4 MB game state is L2-resident by
design.

  value     whole-job env-steps/s, actions resident in HBM, CUDA-event timed
  e2e       the same through SkillshotEnvs.step_host: pinned HOST actions in, the
            step's result back to pinned HOST memory as one packed byte per env-step
            (done, winner, hit tick), copies inside the timing; the three-array form
            (reward / done / winner, 10 B per env-step) is reported beside it
  roofline  HBM: algorithmic 202 B per env-step (SURVEY.md 8(d)) x env-steps per
            launch / average launch time, against MEASURED_PEAKS.json hbm_gbs
  cpu_baseline  the C oracle port (oracle/skillshot_oracle.c, OpenMP over envs)
            on the host cores, on a bounded sample of the same workload, and beside
            it the UNMODIFIED Python reference (oracle/_ref byte-code, one game per
            process over the same cores): env-steps/s in total and per core

  learner   the other half of BASELINE.json's metric, on the same GPUs in the same run:
            rollout (configs[2]: 262,144 envs per GPU, tensor-core actor forward with
            parameter noise + env step with observations + replay push) in env-steps/s and
            samples/s, the DDPG update (sample, TD targets, critic step, actor step, one
            gradient all-reduce each) in update samples/s, and the tensor roofline of the
            actor-forward kernel (72,192 algorithmic FLOP per row against bf16_tflops)

--impl reference times that CPU port alone on all host cores, on the GPU arm's
own config (same keys, same ticks per step), and prints the same line with
"impl": "reference"; the Python reference's figure rides along as
cpu_baseline.python_reference (the port is ~100x faster per core than the Python
objects and is therefore the stricter baseline for the driver's ratio).

--dump-outputs DIR writes, after the timed steps, what the timed path computed in
its last step as DIR/<name>.npy (float32 / float64; at most DUMP_STEP_BYTES of sampled
step outputs plus the game state of every env; see dump_outputs).  The inputs are
seeded, so two builds run with the same arguments can be compared output for output.

Thread counts come from the process's CPU affinity, never from OMP_NUM_THREADS
(torch.distributed.run exports OMP_NUM_THREADS=1).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np

# the CPUs this process may run on, taken BEFORE any NUMA binding of the GPU arm and independent of OMP_NUM_THREADS
# (torch.distributed.run exports OMP_NUM_THREADS=1: the CPU legs must not inherit that)
HOST_CPUS = sorted(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else list(range(os.cpu_count() or 1))


def host_cores() -> int:
    return max(1, len(HOST_CPUS))


class all_host_cpus:
    """Context: run on every CPU the process started with (undo the GPU arm's NUMA binding for the CPU legs)."""

    def __enter__(self):
        self.saved = os.sched_getaffinity(0)
        try:
            os.sched_setaffinity(0, HOST_CPUS)
        except OSError:
            pass
        return self

    def __exit__(self, *exc):
        try:
            os.sched_setaffinity(0, self.saved)
        except OSError:
            pass
        return False


ENVS_PER_GPU = 65536
TICKS = 2048                # ticks per bench step (one full 2,000-tick episode plus the auto-reset)
TICKS_PER_LAUNCH = 1024     # fused ticks per ss_env_step launch (65,536 envs, graph-replayed, tools/explore_step.py: 32: 7.4e10, 128: 8.15e10,
                            # 256: 8.36e10, 512: 8.47e10, 1024: 8.53e10 env-steps/s; a step of 2,048 ticks is two launches)
E2E_TICKS_PER_LAUNCH = 32   # the host-buffer leg pipelines copy in / kernel / copy out per chunk: finer chunks overlap better
TICK_LIMIT = 2000           # SkillshotLearner.py:62
ALGO_BYTES_PER_ENV_STEP = 202   # SURVEY.md 8(d), physics-only
METRIC = "env_steps_per_sec"
UNIT = "env-steps/s"
WORKLOAD = "physics-only: 65,536 SkillshotGame envs per GPU, random actions, terminal reward, 2000-tick auto-reset"


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)), "measured"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


def ncu_profile(ticks_per_launch=None):
    """Per-launch figures of the dominant kernel from the committed `ncu --set full` capture (taken at the default number of
    fused ticks per launch): profiles/traffic.json, or {} when the capture does not match this run."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            t = json.load(open(p))
            if ticks_per_launch is None or t.get("ticks_per_launch", ticks_per_launch) == ticks_per_launch:
                return t
        except Exception:
            pass
    return {}


def ncu_traffic(ticks_per_launch=None):
    """dram bytes per launch of the dominant kernel from that capture, or None."""
    return ncu_profile(ticks_per_launch).get("step_kernel_physics_bytes_per_launch")


def probe_rates(dev):
    """Measured instruction-rate ceilings of this GPU (ss_probe_rates): warp-instructions/s of an alternating LOP3 / IMAD
    stream (the warp schedulers' issue ceiling: two half-rate pipes fed in alternate cycles) and of a DFMA stream (the
    float64 pipe)."""
    import ctypes
    import torch
    from skillshot_learning_b200._lib import lib, check
    out = (ctypes.c_double * 4)()
    scratch = torch.zeros(16, dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        check(lib.ss_probe_rates(out, scratch.data_ptr(), torch.cuda.current_stream(dev).cuda_stream), "ss_probe_rates")
    return {"issue_warp_inst_per_sec": out[0], "fp64_warp_inst_per_sec": out[1], "sms": int(out[2])}


def one_tick_leg(envs, actions, dev, per_graph=64, reps=20):
    """The step kernel at ONE tick per launch on the bench's 65,536 envs: the shape the 202 B per env-step model of
    SURVEY.md 8(d) describes literally (state read and written every tick).  `per_graph` launches are captured in a CUDA
    graph and replayed, so the figure is launch-to-launch time on the device without interpreter time.  Returns seconds
    per launch.  (A replay repeats the captured Philox reset counters: a timing leg, not a trajectory.)"""
    import torch
    s = torch.cuda.Stream(dev)
    with torch.cuda.stream(s):
        for j in range(3):
            envs.step(actions[j], want_obs=False)
        torch.cuda.synchronize(dev)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            for j in range(per_graph):
                envs.step(actions[j % actions.shape[0]], want_obs=False)
        g.replay()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(s)
        for _ in range(reps):
            g.replay()
        e1.record(s)
        torch.cuda.synchronize(dev)
    envs._out = {}
    return e0.elapsed_time(e1) * 1e-3 / (reps * per_graph)


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons during the timed region (NVML)."""

    def __init__(self, index: int, period: float = 0.002):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._halt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
        }
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._halt.set()
        if self.is_alive():
            self.join(timeout=1.0)
        med = int(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ---------------------------------------------------------------------------
# CPU port (oracle) timing -- cpu_baseline leg and --impl reference arm
# ---------------------------------------------------------------------------
def cpu_port_run(n_envs: int, ticks: int, nthreads: int, seed: int = 0, envs=None, actions=None):
    """Times `ticks` ticks of n_envs oracle envs; returns (seconds, envs, actions)."""
    from oracle.oracle import OracleEnvs
    rng = np.random.default_rng(seed)
    if envs is None:
        envs = OracleEnvs(n_envs, rng.integers(25, 225, size=(n_envs, 4)))
    if actions is None:
        actions = rng.uniform(-1.2, 1.2, size=(8, n_envs, 2, 2)).astype(np.float32)
    t0 = time.perf_counter()
    for t in range(ticks):
        envs.step(actions[t % actions.shape[0]], want_obs=False, reward_mode=2, tick_limit=TICK_LIMIT,
                  auto_reset=True, nthreads=nthreads)
    return time.perf_counter() - t0, envs, actions


def python_reference_rate(seconds: float = 2.0):
    """The UNMODIFIED Python reference (SURVEY.md 8(d) config 1) on the host cores: one SkillshotGame per process,
    SkillshotLearner.do_actions for both players + game_tick per env-step.  Runs oracle/py_ref_bench.py as a subprocess
    (no CUDA context is forked) from /root/reference or its byte-code in oracle/_ref.  None when neither exists."""
    import subprocess
    from oracle import ref_harness
    if not ref_harness.available():
        return {"unavailable": "neither /root/reference nor oracle/_ref (python -m oracle.build_ref) on this machine"}
    env = dict(os.environ)
    env.pop("OMP_NUM_THREADS", None)
    try:
        with all_host_cpus():
            out = subprocess.run([sys.executable, "-m", "oracle.py_ref_bench", "--seconds", str(seconds), "--procs", str(host_cores())],
                                 cwd=ROOT, env=env, capture_output=True, text=True, timeout=120)
        rec = json.loads(out.stdout.strip().splitlines()[-1])
    except Exception as e:                                   # the figure is informative: never fail the bench over it
        return {"unavailable": "py_ref_bench failed: %r" % (e,)}
    return {"env_steps_per_sec": rec["tick"]["env_steps_per_sec"], "env_steps_per_sec_per_core": rec["tick"]["env_steps_per_sec_per_core"],
            "with_get_state_prepare_states_env_steps_per_sec": rec["tick_get_state_prepare_states"]["env_steps_per_sec"],
            "cores": rec["procs"], "kind": "reference", "source": rec["source"],
            "sample": "%d processes x one reference SkillshotGame, %.1f s each: do_actions x 2 + game_tick per env-step, "
                      "game_reset(random_positions=True) at a hit or at %d ticks" % (rec["procs"], rec["tick"]["seconds"], TICK_LIMIT)}


def cpu_baseline(target_seconds: float = 4.0):
    """Oracle port on all host cores, bounded sample (~10-30 s of CPU work), the Python reference beside it."""
    cores = host_cores()
    with all_host_cpus():
        _, envs, actions = cpu_port_run(ENVS_PER_GPU, 32, cores)            # cold: thread pool, page faults
        dt, _, _ = cpu_port_run(ENVS_PER_GPU, 32, cores, envs=envs, actions=actions)      # calibration
        ticks = int(max(8, min(4096, target_seconds / max(dt / 32, 1e-6))))
        dt, _, _ = cpu_port_run(ENVS_PER_GPU, ticks, cores, envs=envs, actions=actions)
        out = {"value": ENVS_PER_GPU * ticks / dt, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": "%d envs x %d ticks (%.1f s wall, %d OpenMP threads = the process's CPU affinity) of the same workload, "
                         "C port of the Python reference (oracle/skillshot_oracle.c)" % (ENVS_PER_GPU, ticks, dt, cores)}
        # SURVEY.md 8(d) config 1, second figure: tick + get_state + prepare_states (the rollout's env side)
        t_obs = max(4, ticks // 8)
        t0 = time.perf_counter()
        for t in range(t_obs):
            envs.step(actions[t % actions.shape[0]], want_obs=True, reward_mode=1, tick_limit=TICK_LIMIT, auto_reset=True, nthreads=cores)
        out["with_observations_env_steps_per_sec"] = ENVS_PER_GPU * t_obs / (time.perf_counter() - t0)
        out["learner_update_batch16"] = cpu_learner_baseline()
    out["python_reference"] = python_reference_rate()
    return out


def cpu_learner_baseline(target_seconds: float = 3.0):
    """The reference's own update on the host: Keras-semantics restatement in torch-CPU (oracle/learner_oracle.py; TensorFlow is
    not installable here), batches of 16 as model_param_batch_size (SkillshotLearner.py:61): critic fit step + actor fit step."""
    import torch
    from oracle import learner_oracle as lo
    rng = np.random.default_rng(0)
    L = lo.LearnerOracle(lo.init_actor(rng), lo.init_critic(rng))
    n = 16 * 64
    s = rng.uniform(0, 1, (n, 12)).astype(np.float32); a = rng.uniform(-1, 1, (n, 2)).astype(np.float32)
    y = -rng.uniform(0, 1, n).astype(np.float32); keep = (rng.uniform(size=(n, 256)) >= 0.2).astype(np.float32)
    order = np.arange(n)
    L.critic_fit(s[:32], a[:32], y[:32], order[:32], keep[:32]); L.actor_fit(s[:32])          # warm-up
    done, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < target_seconds:
        L.critic_fit(s, a, y, order, keep)
        L.actor_fit(s)
        done += n
    dt = time.perf_counter() - t0
    return {"samples_per_sec": done / dt, "threads": int(torch.get_num_threads()),
            "sample": "%d rows in batches of 16 (%.1f s): critic fit step + actor fit step per batch, torch-CPU restatement of "
                      "the Keras update (the reference's TensorFlow is not installable here)" % (done, dt)}


ROLLOUT_ENVS = 262144          # BASELINE.json configs[2]
TRAIN_BATCH = 65536            # update rows per GPU per step
SM_BATCH = 148 * 512           # the same sized to the machine: 4 tiles of 128 rows per SM, no partial round
ACTOR_FLOP_PER_ROW = 72192     # SURVEY.md 8(d): 2 * (12*256 + 256*128 + 128*2)
UPDATE_FLOP_PER_ROW = 638976   # SURVEY.md 8(d): full DDPG update with target actor + critic forward on s'


LEG_KEYS = ("roll", "upd", "fwd", "upd32", "upd_big", "cfg5", "upd_sm", "cfg4", "upd_local", "cfg4_solo", "cfg5_upd")
FRAMES5, FRAMES5_BATCH = 20, 65536
# algorithmic FLOP per row of a full DDPG update of the frame-stacked networks: SURVEY.md 8(d)'s 638,976 for 12 inputs plus
# the wider first layers: 12 (F - 1) x 256 more MACs in each of 7 GEMMs (critic forward + dW1; actor-step actor forward,
# critic forward, actor dW1; target actor and critic forward), 2 FLOP per MAC
FRAMES5_UPDATE_FLOP_PER_ROW = UPDATE_FLOP_PER_ROW + 14 * 12 * (FRAMES5 - 1) * 256


def peer_check(dev, rank, world):
    """N > 1: the fused NVLink peer exchange against the NCCL all-reduce on identical seeded minibatches (3 critic + 3 actor
    steps, tensor-core kernels, Philox dropout), and every rank's parameters compared bit for bit.  Raises on a mismatch."""
    import torch
    import torch.distributed as dist
    from skillshot_learning_b200 import ActorCritic
    nets = {c: ActorCritic(device=dev, seed=5, gamma=0.9, tau=0.1, process_group=True, update_precision="bf16", collective=c)
            for c in ("nccl", "peer")}
    start = nets["peer"].params.clone()
    g = torch.Generator(device=dev).manual_seed(77)            # the same data on every rank; each takes its own shard
    n_local = 2048
    n = n_local * world
    sl = slice(rank * n_local, (rank + 1) * n_local)
    for _ in range(3):
        s = torch.rand((n, 12), device=dev, generator=g)
        a = torch.rand((n, 2), device=dev, generator=g) * 2 - 1
        r = -torch.rand(n, device=dev, generator=g)
        for ac in nets.values():
            ac.critic_step(s[sl], a[sl], r[sl])
            ac.actor_step(s[sl])
    nets["peer"].peer.check_status()
    p_peer, p_nccl = nets["peer"].params, nets["nccl"].params
    moved = float((p_peer - start).abs().max())
    diff = float((p_peer - p_nccl).abs().max())
    gathered = [torch.empty_like(p_peer) for _ in range(world)]
    dist.all_gather(gathered, p_peer)
    identical = all(torch.equal(gathered[0], x) for x in gathered)
    nets["peer"].peer.close()
    # Adam turns a last-bit difference of a near-zero gradient into a visible step: the bound is relative to the distance moved
    ok = identical and moved > 0 and diff <= 0.02 * moved + 2e-6
    rec = {"ranks_bit_identical": bool(identical), "peer_vs_nccl_max_abs_diff": diff, "max_param_move": moved, "updates": 3,
           "rows_per_rank": n_local}
    if not ok:
        raise SystemExit("bench.py: multi-GPU peer check FAILED on rank %d: %r" % (rank, rec))
    return rec


def learner_legs(dev, rank, world, seed, peaks, collective, ticks=64, updates=20):
    """Rollout, DDPG update and the actor-forward tensor roofline on this rank's GPU.
    Returns ({leg: ms on this rank}, per-rank check record).  At N > 1 two more legs give the in-run scaling baselines:
    `upd_local` (the same update without the gradient exchange) and `cfg4_solo` (rank 0 alone plays all 1,048,576 envs)."""
    import torch
    import torch.distributed as dist
    from skillshot_learning_b200 import SelfPlayTrainer

    E = ROLLOUT_ENVS
    group = -(-(2 * E // 128) // 148) * 128       # one parameter-noise draw per SM-sized slice of the batch (28 tiles)
    tr = SelfPlayTrainer(E, device=dev, seed=seed, replay_capacity=2 * E * 4, batch_size=TRAIN_BATCH,
                         gamma=0.99, tau=0.005, param_noise_sd=0.5, noise_group=group, reward_mode="looking",
                         tick_limit=TICK_LIMIT, process_group=True if world > 1 else None, precision="bf16",
                         collective=collective)
    t = {k: 0.0 for k in LEG_KEYS}
    checks = {}

    def timed(fn, iters, warm=3):
        for _ in range(warm):
            fn()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1) / iters

    chunk = 16                                     # ticks enqueued per library call (ss_selfplay_rollout)
    t["roll"] = timed(lambda: tr.rollout(chunk), max(1, ticks // chunk)) / chunk
    t["upd"] = timed(tr.update, updates)              # gradient GEMMs on tcgen05 (bf16 operands, f32 accumulate)
    net = tr.networks
    if world > 1:
        # every rank has applied the same summed gradients: the parameters must be bit-identical everywhere
        gathered = [torch.empty_like(net.params) for _ in range(world)]
        dist.all_gather(gathered, net.params)
        checks["trainer_ranks_bit_identical"] = all(torch.equal(gathered[0], x) for x in gathered)
        if net.peer is not None:
            net.peer.check_status()
        if not checks["trainer_ranks_bit_identical"]:
            raise SystemExit("bench.py: ranks diverged after %d sharded updates (rank %d)" % (updates + 3, rank))
        # the same update WITHOUT the exchange (local reduction + Adam): the in-run baseline of the update leg's scaling.
        # It makes the ranks' weights differ, so the learner state is put back afterwards.
        saved = {k: getattr(net, k).clone() for k in ("params", "target", "adam_m", "adam_v")}
        steps = (net.step_actor, net.step_critic)
        grp, peer = net.group, net.peer
        net.group, net.peer, net._update_args = None, None, None
        t["upd_local"] = timed(tr.update, updates)
        net.group, net.peer, net._update_args = grp, peer, None
        for k, v in saved.items():
            getattr(net, k).copy_(v)
        net.step_actor, net.step_critic = steps
    net.update_precision = "f32"
    t["upd32"] = timed(tr.update, max(3, updates // 4))  # the exact float32 kernels, same schedule
    net.update_precision = "bf16"
    tr.batch_size, tr._batch = 2 * E, None            # one update on as many rows as one rollout tick produces
    t["upd_big"] = timed(tr.update, max(3, updates // 2))
    tr.batch_size, tr._batch = SM_BATCH, None         # a whole number of 128-row tiles on every SM
    t["upd_sm"] = timed(tr.update, updates)
    tr.batch_size, tr._batch = TRAIN_BATCH, None
    obs, act = tr.obs.view(-1, 12), tr.actions.view(-1, 2)
    t["fwd"] = timed(lambda: net.actor_forward(obs, out=act, precision="bf16"), 50)
    tr.envs.check_status()
    if net.peer is not None:
        net.peer.check_status()

    # ---- BASELINE.json configs[4]: 20-frame planning actor + randomised per-env game speeds ----
    from skillshot_learning_b200 import FrameStackActor, SkillshotEnvs
    E5, F5 = 65536, 20
    envs5 = SkillshotEnvs(E5, device=dev, random_positions=True, seed=seed + 7, reward_mode="looking", tick_limit=TICK_LIMIT,
                          auto_reset=True)
    g5 = torch.Generator(device=dev).manual_seed(seed + 8)
    scale = lambda: 0.5 + 1.5 * torch.rand(E5, device=dev, generator=g5)          # U(0.5, 2) x the reference constants
    envs5.set_speeds(3.0 * scale(), 0.25 * scale(), 5.0 * scale(), (15.0 * scale()).round().clamp(min=1))
    actor5 = FrameStackActor(2 * E5, frames=F5, device=dev, seed=seed, precision="bf16")
    actor5.push(envs5.observe().reshape(-1, 12))
    act5 = torch.empty((E5, 2, 2), dtype=torch.float32, device=dev)

    def tick5():
        actor5.forward(param_noise_sd=0.5, noise_group=1024, out=act5.view(-1, 2))
        out = envs5.step(act5)
        actor5.push(out["obs"].reshape(-1, 12), out["done"], done_div=2)

    t["cfg5"] = timed(tick5, 32)
    envs5.check_status()
    # ... and its learner: the DDPG update of the 240-input actor and critic (float32 kernels, separate steps) on a
    # minibatch drawn from a ring of stacked observations that a short self-play rollout has filled
    del envs5, actor5
    torch.cuda.empty_cache()
    tr5 = SelfPlayTrainer(16384, device=dev, seed=seed + 9, frames=F5, batch_size=FRAMES5_BATCH, replay_capacity=2 * 16384 * 4,
                          gamma=0.99, tau=0.005, param_noise_sd=0.5, noise_group=1024, reward_mode="looking",
                          tick_limit=TICK_LIMIT, precision="bf16", process_group=True if world > 1 else None, collective=collective)
    tr5.rollout(4)
    t["cfg5_upd"] = timed(tr5.update, 4, warm=1)
    tr5.envs.check_status()
    if tr5.networks.peer is not None:
        tr5.networks.peer.check_status()
        tr5.networks.peer.close()
    del tr5

    # ---- BASELINE.json configs[3]: full self-play training, 1,048,576 envs in total sharded over the GPUs ----
    if tr.networks.peer is not None:
        tr.networks.peer.close()
    del tr
    torch.cuda.empty_cache()

    def config4(n_envs, group, coll):
        tr4 = SelfPlayTrainer(n_envs, device=dev, seed=seed + 11, replay_capacity=2 * n_envs * 2, batch_size=TRAIN_BATCH,
                              process_group=group, gamma=0.99, tau=0.005, param_noise_sd=0.5,
                              noise_group=-(-(2 * n_envs // 128) // 148) * 128, reward_mode="looking", tick_limit=TICK_LIMIT,
                              precision="bf16", collective=coll)

        def iteration():
            tr4.rollout(1)
            tr4.update()

        return tr4, iteration

    tr4, iteration = config4(1048576 // world, True if world > 1 else None, collective)
    t["cfg4"] = timed(iteration, 16)
    tr4.envs.check_status()
    if tr4.networks.peer is not None:
        tr4.networks.peer.check_status()
        tr4.networks.peer.close()
    del tr4, iteration
    torch.cuda.empty_cache()
    if world > 1:
        # strong-scaling baseline measured in the same run: rank 0 alone plays the whole 1,048,576 envs, the others wait
        if rank == 0:
            tr1, it1 = config4(1048576, None, "nccl")
            for _ in range(3):
                it1()
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(16):
                it1()
            e1.record()
            torch.cuda.synchronize(dev)
            t["cfg4_solo"] = e0.elapsed_time(e1) / 16
            del tr1, it1
            torch.cuda.empty_cache()
        dist.barrier()
        if collective == "peer":
            checks["peer_vs_nccl"] = peer_check(dev, rank, world)
    return t, checks


def learner_report(t, world, peaks, peak_kind, collective="nccl", t_min=None):
    """The `learner` object of the line from the per-leg times (ms, max over ranks; t_min: min over ranks)."""
    rows = 2 * ROLLOUT_ENVS
    t_roll, t_upd, t_fwd, t_upd32, t_upd_big, t_cfg5, t_upd_sm, t_cfg4 = (t[k] for k in LEG_KEYS[:8])
    tf = ACTOR_FLOP_PER_ROW * rows / (t_fwd * 1e-3) / 1e12
    rep = {
        "rollout": {"workload": "262,144 envs per GPU: bf16 tensor-core actor forward on 524,288 observations with "
                                "parameter noise (sd 0.5) + env step with observations and looking reward, transitions produced "
                                "in place in the replay ring; 16 ticks per ss_selfplay_rollout call",
                    "env_steps_per_sec": world * ROLLOUT_ENVS / (t_roll * 1e-3),
                    "samples_per_sec": world * rows / (t_roll * 1e-3), "ms_per_tick": t_roll},
        "train": {"workload": "DDPG update, %d rows per GPU: replay sample, TD targets (gamma 0.99), critic step "
                              "(dropout 0.2), actor step, Adam + soft update (tau 0.005), two flat-gradient exchanges (%s)"
                              % (TRAIN_BATCH, "single GPU: none" if world == 1 else
                                 ("fused NVLink peer-memory reduce-push + Adam" if collective == "peer" else "NCCL all-reduce")),
                  "samples_per_sec": world * TRAIN_BATCH / (t_upd * 1e-3), "ms_per_update": t_upd,
                  "dtype": "bf16 operands, f32 accumulate (tcgen05); Adam and parameters f32",
                  "algorithmic_tflops": world * TRAIN_BATCH * UPDATE_FLOP_PER_ROW / (t_upd * 1e-3) / 1e12,
                  "tensor_frac": TRAIN_BATCH * UPDATE_FLOP_PER_ROW / (t_upd * 1e-3) / 1e12 / peaks["bf16_tflops"],
                  "f32_path_samples_per_sec": world * TRAIN_BATCH / (t_upd32 * 1e-3),
                  "rows_75776_per_gpu": {"note": "148 SMs x 512 rows: every SM gets 4 whole tiles (65,536 rows are 3.46 per SM, "
                                                 "i.e. 4 rounds with a partial one)",
                                         "samples_per_sec": world * SM_BATCH / (t_upd_sm * 1e-3), "ms_per_update": t_upd_sm,
                                         "algorithmic_tflops": world * SM_BATCH * UPDATE_FLOP_PER_ROW / (t_upd_sm * 1e-3) / 1e12},
                  "rows_524288_per_gpu": {"samples_per_sec": world * rows / (t_upd_big * 1e-3), "ms_per_update": t_upd_big,
                                          "algorithmic_tflops": world * rows * UPDATE_FLOP_PER_ROW / (t_upd_big * 1e-3) / 1e12,
                                          "tensor_frac": rows * UPDATE_FLOP_PER_ROW / (t_upd_big * 1e-3) / 1e12 / peaks["bf16_tflops"]}},
        "selfplay_training": {
            "workload": "BASELINE.json configs[3]: 1,048,576 envs in total (%d per GPU), one iteration = one rollout tick of every env "
                        "(tensor-core actor, parameter noise, transitions into the replay ring) + one %d-row-per-GPU DDPG update; "
                        "strong scaling (the total is fixed)" % (1048576 // world, TRAIN_BATCH),
            "env_steps_per_sec": 1048576 / (t_cfg4 * 1e-3), "update_samples_per_sec": world * TRAIN_BATCH / (t_cfg4 * 1e-3),
            "ms_per_iteration": t_cfg4},
        "planning_actor_speed_sweep": {
            "workload": "BASELINE.json configs[4] (no reference code): 65,536 envs per GPU with per-env speed constants "
                        "U(0.5, 2) x the reference's, 20-frame stacked-observation actor (240 -> 256 -> 128 -> 2, tcgen05 "
                        "kernels) with parameter noise (sd 0.5, one draw per 1,024 rows) + env step + frame-stack push",
            "env_steps_per_sec": world * 65536 / (t_cfg5 * 1e-3), "samples_per_sec": world * 131072 / (t_cfg5 * 1e-3),
            "ms_per_tick": t_cfg5,
            "train": {"workload": "DDPG update of the 20-frame networks (actor 240 -> 256 -> 128 -> 2, critic 240 -> 256 -> (+2) -> "
                                  "128 -> 1), %d rows per GPU drawn from a ring of stacked observations: TD targets, critic step "
                                  "(dropout 0.2), actor step, Adam + soft update; exact float32 kernels (CUDA cores), separate steps"
                                  % FRAMES5_BATCH,
                      "samples_per_sec": world * FRAMES5_BATCH / (t["cfg5_upd"] * 1e-3) if t.get("cfg5_upd") else None,
                      "ms_per_update": t.get("cfg5_upd"),
                      "algorithmic_flop_per_row": FRAMES5_UPDATE_FLOP_PER_ROW,
                      "algorithmic_tflops": (world * FRAMES5_BATCH * FRAMES5_UPDATE_FLOP_PER_ROW / (t["cfg5_upd"] * 1e-3) / 1e12
                                             if t.get("cfg5_upd") else None),
                      "tensor_frac": (FRAMES5_BATCH * FRAMES5_UPDATE_FLOP_PER_ROW / (t["cfg5_upd"] * 1e-3) / 1e12 / peaks["bf16_tflops"]
                                      if t.get("cfg5_upd") else None),
                      "dtype": "f32 (no tensor cores on this leg: the fraction is against the bf16 tensor peak for comparison)"}},
        "actor_forward_roofline": {"bound": "tensor", "achieved": tf, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
                                   "frac": tf / peaks["bf16_tflops"], "traffic": None, "peak_source": peak_kind,
                                   "kernel": "actor_fwd_tc_kernel", "rows_per_launch": rows,
                                   "algorithmic_flop_per_row": ACTOR_FLOP_PER_ROW, "launch_us": t_fwd * 1e3,
                                   "dtype": "bf16 operands, f32 accumulate"},
    }
    if world > 1:
        # Per-leg scaling measured INSIDE this run (the driver computes the headline's efficiency itself from its 1/2/4/8 runs):
        #   update     the same update without the exchange (local reduction + Adam) / the sharded update: the cost of the two exchanges
        #   config 4   strong scaling: rank 0 alone on all 1,048,576 envs / (N x the sharded iteration)
        #   rollout    no exchange on this leg: fastest rank / slowest rank of the concurrent run
        sc = {"update_weak_efficiency": t["upd_local"] / t_upd if t.get("upd_local") else None,
              "update_ms_without_exchange": t.get("upd_local") or None,
              "config4_strong_speedup": t["cfg4_solo"] / t_cfg4 if t.get("cfg4_solo") else None,
              "config4_strong_efficiency": t["cfg4_solo"] / t_cfg4 / world if t.get("cfg4_solo") else None,
              "config4_ms_per_iteration_one_gpu_all_envs": t.get("cfg4_solo") or None}
        if t_min is not None:
            sc["rollout_fastest_over_slowest_rank"] = t_min["roll"] / t_roll
            sc["planning_actor_fastest_over_slowest_rank"] = t_min["cfg5"] / t_cfg5
        rep["scaling_in_run"] = sc
    return rep


def bench_config(ticks: int, ticks_per_launch: int) -> dict:
    """The `config` object of the line -- the same in both arms (the driver compares them)."""
    return {"workload": WORKLOAD, "envs_per_gpu": ENVS_PER_GPU, "ticks_per_step": ticks, "ticks_per_launch": ticks_per_launch,
            "l2": "action stream per step (%.0f MB) exceeds the 126 MB L2; game state (4 MB) is L2-resident by design"
                  % (ticks * ENVS_PER_GPU * 16 / 1e6)}


def run_reference_arm(args):
    """The reference's CPU implementation of the path on the host cores, on the GPU arm's config: each step is
    `ticks_per_step` ticks of 65,536 envs (the C port steps tick by tick; `ticks_per_launch` is the GPU arm's launch
    granularity and has no CPU counterpart).  Rank 0 alone runs it, on every core of the box."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = host_cores()
    T = args.ticks
    _, envs, actions = cpu_port_run(ENVS_PER_GPU, 64, cores)                     # cold: thread pool, page faults
    dt, _, _ = cpu_port_run(ENVS_PER_GPU, 64, cores, envs=envs, actions=actions)
    dt /= 8
    # bounded sample: a step is the first `sample_ticks` ticks of the config's step when the whole step would not fit ~3 minutes
    budget = 150.0 / max(1, args.steps + args.warmup)
    sample_ticks = T
    while sample_ticks > 64 and (dt / 8) * sample_ticks > budget:
        sample_ticks //= 2
    for _ in range(args.warmup):
        cpu_port_run(ENVS_PER_GPU, sample_ticks, cores, envs=envs, actions=actions)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_port_run(ENVS_PER_GPU, sample_ticks, cores, envs=envs, actions=actions)
    dt = time.perf_counter() - t0
    value = ENVS_PER_GPU * sample_ticks * args.steps / dt
    sample = ("each step = %d envs x %d of the step's %d ticks on %d OpenMP threads (CPU affinity of the process; OMP_NUM_THREADS=%s "
              "ignored); C port of the Python reference" % (ENVS_PER_GPU, sample_ticks, T, cores, os.environ.get("OMP_NUM_THREADS", "unset")))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps * (T / sample_ticks),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": bench_config(T, args.ticks_per_launch),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                         "python_reference": python_reference_rate()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


DUMP_STEP_BYTES = 32 << 20     # --dump-outputs: bound on the sampled step outputs (16 B per env-tick as float32)


def dump_outputs(path: str, envs, out: dict):
    """--dump-outputs: what the timed path handed its caller in its last step, written as path/<name>.npy.
    SkillshotEnvs.step reuses its output tensors from launch to launch, so once a step has returned its caller holds the
    reward / done / winner of the step's last launch [ticks_per_launch, envs, ...]: those of every tick for as many env
    columns as fit DUMP_STEP_BYTES, drawn with a fixed seed (their indices in env_index), as float32.  The step's earlier
    launches are not in these buffers any more: they show only through the game state every env is left in after the
    step (SkillshotEnvs.export_state, state_<field>), written beside them as float64."""
    import torch
    os.makedirs(path, exist_ok=True)
    ticks = out["reward"].shape[0]
    n_cols = max(1, min(envs.n_envs, DUMP_STEP_BYTES // (16 * ticks)))
    cols = np.sort(np.random.default_rng(0).choice(envs.n_envs, n_cols, replace=False))
    idx = torch.from_numpy(cols).to(out["reward"].device)
    arrays = {"env_index": cols.astype(np.float64)}
    for k in ("reward", "done", "winner"):
        arrays[k] = out[k].index_select(1, idx).cpu().numpy().astype(np.float32)
    for k, v in envs.export_state().items():
        arrays["state_" + k] = np.asarray(v, dtype=np.float64)
    for k, v in arrays.items():
        np.save(os.path.join(path, k + ".npy"), v)


def bind_to_gpu_numa(index: int):
    """Pin this process to the CPUs NVML reports as local to GPU `index`, BEFORE the pinned host buffers of the
    end-to-end leg are allocated (first touch then lands on the GPU's own NUMA node).  With 8 ranks streaming
    3.5 GB per step each through host memory, remote-socket buffers halve the end-to-end rate."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (m >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return 0


# ---------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------
def run_gpu_arm(args):
    import torch
    import torch.distributed as dist
    from skillshot_learning_b200 import SkillshotEnvs

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the GPU arm has no CPU fallback)")
    numa_cpus = bind_to_gpu_numa(local)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    E, T, KF = ENVS_PER_GPU, args.ticks, args.ticks_per_launch
    assert T % KF == 0
    launches_per_step = T // KF
    envs = SkillshotEnvs(E, device=dev, random_positions=True, seed=1234 + rank, reward_mode="terminal",
                         tick_limit=TICK_LIMIT, auto_reset=True)
    gen = torch.Generator(device=dev)
    gen.manual_seed(99 + rank)
    actions = (torch.rand((T, E, 2, 2), device=dev, generator=gen) * 2.4 - 1.2).contiguous()

    def device_step():
        for c in range(launches_per_step):
            out = envs.step(actions[c * KF:(c + 1) * KF], want_obs=False)
        return out

    # ---- device-resident throughput (value) ----
    for _ in range(max(args.warmup, 3)):
        device_step()
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        out = device_step()
    ev1.record()
    barrier()
    clocks = sampler.stop()
    ms = ev0.elapsed_time(ev1)
    envs.check_status()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, envs, out)

    # ---- the same kernel family at one tick per launch (the literal 202 B per env-step shape), and the GPU's measured
    #      instruction-rate ceilings for the record of the bound the fused kernel is actually on ----
    one_tick_s = one_tick_leg(envs, actions, dev) if rank == 0 else 0.0
    rates = probe_rates(dev) if rank == 0 else None
    barrier()

    # ---- end to end through the host-buffer API (e2e) ----
    e2e_steps, e2e_s, e2e_solo_s, e2e_solo_steps, e2e_flags_s = max(3, min(args.steps, 10)), float("nan"), 0.0, 3, float("nan")
    KE = E2E_TICKS_PER_LAUNCH if T % E2E_TICKS_PER_LAUNCH == 0 else KF
    if not args.no_e2e:
        host_actions = torch.empty((T, E, 2, 2), dtype=torch.float32, pin_memory=True)
        host_actions.copy_(actions)
        host_out = envs.alloc_host_outputs(T)
        for _ in range(2):
            envs.step_host(host_actions, host_out, ticks_per_launch=KE)
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            envs.step_host(host_actions, host_out, ticks_per_launch=KE)   # synchronises before returning
        barrier()
        e2e_s = time.perf_counter() - t0
        # the same with the packed one-byte-per-env-step output (ss_env_step_packed: done, winner and the tick of the hit, from
        # which the terminal reward follows): 17 B per env-step cross the bus instead of 26
        flags_out = envs.alloc_host_outputs(T, outputs="flags")
        envs.step_host(host_actions, flags_out, ticks_per_launch=KE)
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            envs.step_host(host_actions, flags_out, ticks_per_launch=KE)
        barrier()
        e2e_flags_s = time.perf_counter() - t0
        if world > 1:
            # in-run baseline of this leg's scaling: rank 0 alone on the host's memory and PCIe fabric, the others idle
            if rank == 0:
                t0 = time.perf_counter()
                for _ in range(e2e_solo_steps):
                    envs.step_host(host_actions, flags_out, ticks_per_launch=KE)
                e2e_solo_s = time.perf_counter() - t0
            barrier()
        del host_actions, host_out, flags_out

    # ---- learner legs: rollout, DDPG update, tensor roofline of the actor forward ----
    lt, checks = {k: float("nan") for k in LEG_KEYS}, {}
    if not args.no_learner:
        del actions
        torch.cuda.empty_cache()
        lt, checks = learner_legs(dev, rank, world, 4321 + rank, measured_peaks()[0], args.collective)

    lt_min = None
    if world > 1:
        t = torch.tensor([ms, e2e_s, e2e_solo_s, e2e_flags_s] + [lt[k] for k in LEG_KEYS], dtype=torch.float64, device=dev)
        tmin = t.clone()
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tmin, op=dist.ReduceOp.MIN)
        ms, e2e_s, e2e_solo_s, e2e_flags_s = float(t[0]), float(t[1]), float(t[2]), float(t[3])
        lt = {k: float(x) for k, x in zip(LEG_KEYS, t[4:])}
        lt_min = {k: float(x) for k, x in zip(LEG_KEYS, tmin[4:])}

    if rank == 0:
        peaks, peak_kind = measured_peaks()
        total_env_steps = world * E * T * args.steps
        value = total_env_steps / (ms * 1e-3)
        launch_s = (ms * 1e-3) / (args.steps * launches_per_step)
        achieved = ALGO_BYTES_PER_ENV_STEP * E * KF / launch_s / 1e9
        prof = ncu_profile(KF)
        traffic = prof.get("step_kernel_physics_bytes_per_launch")
        inst = prof.get("step_kernel_physics_warp_inst_per_launch")
        fp64_inst = prof.get("step_kernel_physics_fp64_warp_inst_per_launch")
        one_tick_gbs = ALGO_BYTES_PER_ENV_STEP * E / one_tick_s / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": bench_config(T, KF),
            # frac follows SURVEY.md 8(d): ALGORITHMIC bytes (202 per env-step) / launch time / measured HBM peak.  The fused
            # kernel plays KF ticks per launch out of registers, so the bytes it really moves are ~1/8 of that: dram_frac is
            # the fraction of the HBM peak its measured DRAM traffic amounts to, and `actual_bound` is the record of the
            # resource it is actually limited by (instruction issue), against ceilings measured on this GPU in this run.
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": achieved / peaks["hbm_gbs"], "traffic": traffic, "peak_source": peak_kind,
                         "kernel": prof.get("kernel", "step_kernel (fused physics ticks)"),
                         "algorithmic_bytes_per_env_step": ALGO_BYTES_PER_ENV_STEP,
                         "moved_bytes_per_env_step": 16 + 8 + 2 + 128.0 / KF,
                         "launch_us": launch_s * 1e6,
                         "dram_achieved": None if traffic is None else traffic / launch_s / 1e9,
                         "dram_frac": None if traffic is None else traffic / launch_s / 1e9 / peaks["hbm_gbs"],
                         "one_tick_per_launch": {
                             "note": "the same 65,536 envs at ONE tick per launch (state read and written every tick: the shape the "
                                     "202 B model describes literally), 64 launches per CUDA-graph replay",
                             "launch_us": one_tick_s * 1e6, "achieved": one_tick_gbs, "frac": one_tick_gbs / peaks["hbm_gbs"],
                             "env_steps_per_sec": E / one_tick_s},
                         "actual_bound": None if rates is None else {
                             "bound": "issue", "unit": "warp-instructions/s",
                             "achieved": None if inst is None else inst / launch_s,
                             "peak": rates["issue_warp_inst_per_sec"],
                             "frac": None if inst is None else inst / launch_s / rates["issue_warp_inst_per_sec"],
                             "warp_instructions_per_launch": inst,
                             "fp64": {"achieved": None if fp64_inst is None else fp64_inst / launch_s,
                                      "peak": rates["fp64_warp_inst_per_sec"],
                                      "frac": None if fp64_inst is None else fp64_inst / launch_s / rates["fp64_warp_inst_per_sec"]},
                             "peak_source": "ss_probe_rates in this run: register-only LOP3+IMAD / DFMA streams (csrc/ss_probe.cu); "
                                            "instruction counts per launch from the committed ncu capture (profiles/traffic.json)"}},
            # SkillshotEnvs.step_host with pinned HOST buffers, copies inside the timed region.  The step's result comes back as
            # one packed byte per env-step (done, winner_id, hit tick: reward / done / winner follow from it without loss,
            # SkillshotEnvs.unpack_flags); the same call returning the three arrays separately (10 B per env-step) is beside it.
            "e2e": {"value": None if args.no_e2e else world * E * T * e2e_steps / e2e_flags_s, "unit": UNIT,
                    "h2d_bytes_per_step": T * E * 16, "d2h_bytes_per_step": T * E,
                    "ticks_per_launch": KE,
                    "outputs": "step_host(outputs='flags'): uint8 [T, E] = done | winner_id << 1 | hit << 3",
                    "note": "bus-bound: 17 B per env-step cross PCIe (16 of float32 actions up, 1 packed result byte down); "
                            "rank processes pinned to their GPU's NUMA node (%d CPUs) before the pinned buffers are allocated"
                            % numa_cpus,
                    "full_outputs": {"value": None if args.no_e2e else world * E * T * e2e_steps / e2e_s, "unit": UNIT,
                                     "d2h_bytes_per_step": T * E * 10,
                                     "note": "the same call returning reward float32 [T,E,2], done and winner uint8 [T,E]: 26 B per "
                                             "env-step on the bus (round 1's e2e figure)"}},
            "gpu_launches": args.steps * launches_per_step,
            "clocks": clocks,
        }
        if world > 1 and not args.no_e2e and e2e_solo_s > 0:
            solo = E * T * e2e_solo_steps / e2e_solo_s
            line["e2e"]["one_rank_alone_env_steps_per_sec"] = solo
            line["e2e"]["weak_efficiency_in_run"] = line["e2e"]["value"] / (world * solo)
        if not args.no_learner:
            line["learner"] = learner_report(lt, world, peaks, peak_kind, args.collective, lt_min)
            if world > 1:
                ok = bool(checks.get("trainer_ranks_bit_identical")) and (args.collective != "peer" or "peer_vs_nccl" in checks)
                line["peer_check"] = "ok" if ok else "failed"
                line["peer_check_detail"] = checks
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline()
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--ticks", type=int, default=TICKS)
    ap.add_argument("--ticks-per-launch", type=int, default=TICKS_PER_LAUNCH)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="profiling runs only: skip the host-buffer leg")
    ap.add_argument("--no-learner", action="store_true", help="skip the rollout / update / actor-forward legs")
    ap.add_argument("--collective", default="peer", choices=["peer", "nccl"],
                    help="gradient exchange of the update at N > 1: fused NVLink peer-memory kernels, or an NCCL all-reduce")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step to DIR/<name>.npy (rank 0's envs): per-tick reward / "
                         "done / winner of the step's last launch for a seeded sample of envs (the step's earlier "
                         "launches show only through the game state) and the game state of every env after the step")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU arm's timed path (--impl b200)")
    if args.impl == "reference":
        return run_reference_arm(args)
    return run_gpu_arm(args)


if __name__ == "__main__":
    sys.exit(main())
