"""Device time of one rollout tick of a trainer that plays part of its envs against a pool of frozen opponents
(SelfPlayTrainer(opponents=...).rollout: learner forward + opponents' segment forward + ss_env_step_pool) against one
self-play rollout tick (ss_selfplay_rollout) at the same env count, alternated in one process and timed with CUDA events.

    python tools/pool_rollout_time.py [--ticks 64] [--rounds 3] [--profile DIR]

Setup of both: bf16 forwards, parameter noise 0.5 in groups of 128 rows, looking reward, random starts, the replay ring
written in place (default capacity, 8 ticks).  Cases at 262,144 envs: M = n / 2 pool envs against K = 8 opponents,
M = n against K = 16, M = 0 (the pool path with no pool envs); and M = n / 2, K = 8 at 65,536 envs.  Each round times one
call of `ticks` ticks per trainer after a warm-up call; a case reports the best of its rounds, per tick.  Prints the card's
name, power limit and SM clocks read in the same run.  --profile DIR writes torch.profiler per-kernel tables of 4 ticks of
the M = n / 2, K = 8 pool trainer and of the self-play trainer at 262,144 envs, a run of its own after the timed ones, with
the launches not chained (ss_set_dependent_launch(0)): a chained grid is placed early and waits for its predecessor, and
the profiler would count that wait as the kernel's time."""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from skillshot_learning_b200 import ActorCritic, SelfPlayTrainer  # noqa: E402
from skillshot_learning_b200._lib import lib  # noqa: E402


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name(0) + ", power limit unknown"


def timed(tr, n_ticks):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    tr.rollout(n_ticks)
    b.record()
    b.synchronize()
    return a.elapsed_time(b) * 1000.0 / n_ticks       # us per tick


def trainer(n, M=None, K=0):
    kw = dict(seed=1, precision="bf16", param_noise_sd=0.5, noise_group=128, reward_mode="looking", tick_limit=2000)
    if K:
        kw.update(opponents=[ActorCritic(seed=10 + k).actor for k in range(K)], pool_envs=M)
    return SelfPlayTrainer(n, **kw)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ticks", type=int, default=64)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--profile", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    print(card())
    cases = [(262144, 131072, 8), (262144, 262144, 16), (262144, 0, 1), (65536, 32768, 8)]
    print("%-34s %12s %14s %7s" % ("case", "pool tick", "self-play tick", "ratio"))
    for n, M, K in cases:
        pool, selfplay = trainer(n, M, K), trainer(n)
        for tr in (pool, selfplay):
            tr.rollout(args.ticks)                   # warm-up: module loads, the ring's first pass
        best_p = best_s = float("inf")
        for _ in range(args.rounds):
            best_p = min(best_p, timed(pool, args.ticks))
            best_s = min(best_s, timed(selfplay, args.ticks))
        print("%-34s %9.1f us %11.1f us %6.3fx" % ("n=%d M=%d K=%d" % (n, M, K), best_p, best_s, best_p / best_s))
        del pool, selfplay
        torch.cuda.empty_cache()
    if args.profile:
        from torch.profiler import ProfilerActivity, profile
        os.makedirs(args.profile, exist_ok=True)
        lib.ss_set_dependent_launch(0)
        for name, tr in (("pool_n2_k8", trainer(262144, 131072, 8)), ("selfplay", trainer(262144))):
            tr.rollout(8)
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                tr.rollout(4)
                torch.cuda.synchronize()
            with open(os.path.join(args.profile, "kernels_%s_262144.txt" % name), "w") as f:
                f.write(card() + "\n4 rollout ticks, 262,144 envs, bf16, launches not chained\n")
                f.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=20, max_name_column_width=70))
            del tr
            torch.cuda.empty_cache()
        lib.ss_set_dependent_launch(1)


if __name__ == "__main__":
    main()
