"""What per-env game speeds cost a pool (SelfPlayTrainer(opponents=...) with envs.set_speeds, ss_env_step_pool_speeds,
ss_pool_rollout_speeds):

  1. the env step alone at 262,144 envs, M = n / 2 pool envs, K = 8 opponents, with a config-5 style speed sweep (each
     constant U(0.5, 2) times the reference's): the pool step with speeds (ss_env_step_pool_speeds) against the self-play
     step with the same speeds (ss_env_step_ring, one tick, observations and their second copy) and the pool step without
     speeds (ss_env_step_pool_blocks), per kernel with torch.profiler, each in a run of its own of `launches` launches;
  2. the whole pool tick (one ss_pool_rollout_speeds / ss_pool_rollout_frames call of `ticks` ticks, timed with CUDA
     events, best of `rounds`, the two trainers alternated) of a trainer with the speed sweep against the same trainer
     without speeds: a 1-frame learner against 8 1-frame opponents at 65,536 and 262,144 envs, and a 20-frame learner
     against 8 20-frame opponents at 65,536 envs, M = n / 2.

    python tools/pool_speeds_time.py [--ticks 32] [--rounds 3] [--launches 100] [--out DIR]

Setup: bf16 forwards, parameter noise 0.5 in groups of 128 rows, looking reward, random starts, episode statistics on,
the replay ring written in place (default capacity, 8 ticks).  Prints the card's name, power limit and SM clocks read in
the same run; --out DIR writes the tables (r8_pool_speeds_step_262144.txt, r8_pool_speeds_time.txt)."""
import argparse
import ctypes
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from skillshot_learning_b200 import ActorCritic, SelfPlayTrainer, SkillshotEnvs  # noqa: E402
from skillshot_learning_b200._lib import lib  # noqa: E402
from skillshot_learning_b200.learner import FrameStackActor  # noqa: E402

K = 8


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name(0) + ", power limit unknown"


def sweep(n, seed):
    """bench.py's configs[4] speeds: each constant U(0.5, 2) times the reference's, the cooldown rounded, at least 1"""
    g = torch.Generator(device="cuda").manual_seed(seed)
    scale = lambda: 0.5 + 1.5 * torch.rand(n, device="cuda", generator=g)
    return 3.0 * scale(), 0.25 * scale(), 5.0 * scale(), (15.0 * scale()).round().clamp(min=1)


def step_kernels(n, launches):
    """per-kernel device time of the three steps (torch.profiler), us per launch"""
    from torch.profiler import ProfilerActivity, profile
    M = n // 2
    L = 2 * n - M
    d = dict(device="cuda")
    g = torch.Generator(device="cuda").manual_seed(0)
    act = torch.rand(2 * n, 2, generator=g, **d) * 2.4 - 1.2
    obs, obs2, reward = torch.empty(2 * n, 12, **d), torch.empty(2 * n, 12, **d), torch.empty(2 * n, **d)
    done_rows, opp_obs = torch.empty(2 * n, dtype=torch.uint8, **d), torch.empty(M, 12, **d)
    done, winner = torch.empty(n, dtype=torch.uint8, **d), torch.empty(n, dtype=torch.uint8, **d)
    status, stats = torch.zeros(2 + 144, dtype=torch.int32, **d), torch.zeros(K, 8, dtype=torch.int64, **d)
    table = (ctypes.c_int64 * K)(*([M // K] * K))
    out, tables = [], []
    for kind, name, kernel in (("pool speeds", "ss_env_step_pool_speeds", "pool_step_speeds_kernel"),
                               ("ring", "ss_env_step_ring, speeds", "step_kernel<"),
                               ("pool", "ss_env_step_pool_blocks, no speeds", "step_pp_obs_kernel")):
        env = SkillshotEnvs(n, random_positions=True, seed=1)
        env.set_speeds(*sweep(n, 2))

        def step(t):
            if kind == "ring":
                rc = lib.ss_env_step_ring(env.state.data_ptr(), n, act.data_ptr(), obs.data_ptr(), obs2.data_ptr(), reward.data_ptr(),
                                          done.data_ptr(), done_rows.data_ptr(), winner.data_ptr(), 1, 1, 2000, 1, 1, 5, t,
                                          env.speeds.data_ptr(), status.data_ptr(), 2, None)
            else:
                args = [env.state.data_ptr(), n, M, K, act.data_ptr(), act[L:].data_ptr(), obs.data_ptr(), obs2.data_ptr(),
                        reward.data_ptr(), done_rows.data_ptr(), opp_obs.data_ptr(), done.data_ptr(), winner.data_ptr(), 1, 2000, 1, 5, t,
                        status.data_ptr(), 2, stats.data_ptr(), table]
                rc = (lib.ss_env_step_pool_speeds(*(args + [env.speeds.data_ptr(), None])) if kind == "pool speeds"
                      else lib.ss_env_step_pool_blocks(*(args + [None])))
            assert rc == 0
        for t in range(20):
            step(t)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for t in range(launches):
                step(100 + t)
            torch.cuda.synchronize()
        ev = [e for e in prof.key_averages() if kernel in e.key]
        assert len(ev) == 1, [e.key for e in prof.key_averages()]
        us = getattr(ev[0], "self_device_time_total", None) or ev[0].self_cuda_time_total
        out.append((name, us / ev[0].count))
        tables.append("== %s ==\n" % name + prof.key_averages().table(sort_by="cuda_time_total", row_limit=6, max_name_column_width=70))
        del env
    return out, tables


def trainer(n, frames, speeds):
    kw = dict(seed=1, precision="bf16", param_noise_sd=0.5, noise_group=128, reward_mode="looking", tick_limit=2000, frames=frames)
    opp = [ActorCritic(seed=10 + k).actor if frames == 1 else FrameStackActor(8, frames=frames, seed=10 + k, device="cuda").params
           for k in range(K)]
    tr = SelfPlayTrainer(n, opponents=opp, pool_envs=n // 2, **kw)
    if speeds:
        tr.envs.set_speeds(*sweep(n, 3))
    return tr


def timed(tr, n_ticks):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    tr.rollout(n_ticks)
    b.record()
    b.synchronize()
    return a.elapsed_time(b) * 1000.0 / n_ticks       # us per tick


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ticks", type=int, default=32)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--launches", type=int, default=100)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    head = card()
    print(head)
    lines = [head]

    steps, tables = step_kernels(262144, args.launches)
    base = steps[1][1]
    lines.append("env step alone, n=262144 M=131072 K=8, speed sweep, %d launches each, torch.profiler (launches not chained); "
                 "ratios against the self-play step with the same speeds" % args.launches)
    for name, us in steps:
        lines.append("%-36s %8.2f us  %6.3fx" % (name, us, us / base))
    print("\n".join(lines[1:]))
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "r8_pool_speeds_step_262144.txt"), "w") as f:
            f.write("\n".join(lines) + "\n\n" + "\n\n".join(tables) + "\n")

    rows = ["%-44s %12s %12s %8s" % ("case", "no speeds", "speeds", "ratio")]
    print(rows[0])
    for n, frames in ((65536, 1), (262144, 1), (65536, 20)):
        M = n // 2
        trs = [trainer(n, frames, False), trainer(n, frames, True)]
        for tr in trs:
            tr.rollout(args.ticks)                   # warm-up: module loads, the ring's first pass
        best = [float("inf")] * 2
        for _ in range(args.rounds):
            for i, tr in enumerate(trs):
                best[i] = min(best[i], timed(tr, args.ticks))
        for tr in trs:
            tr.envs.check_status()
        row = "%-44s %9.1f us %9.1f us %7.3fx" % ("n=%d M=%d K=8 x %d frames (learner %d)" % (n, M, frames, frames), best[0], best[1],
                                                  best[1] / best[0])
        print(row)
        rows.append(row)
        del trs, tr
        torch.cuda.empty_cache()
    if args.out:
        with open(os.path.join(args.out, "r8_pool_speeds_time.txt"), "w") as f:
            f.write(head + "\npool tick per trainer (one ss_pool_rollout_frames / ss_pool_rollout_speeds call of %d ticks, best of %d "
                    "rounds, alternated); ratio: with the speed sweep over without speeds\n" % (args.ticks, args.rounds) +
                    "\n".join(rows) + "\n")


if __name__ == "__main__":
    main()
