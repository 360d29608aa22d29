"""What pool blocks of any size per opponent cost (SelfPlayTrainer(opponents=...).set_pool_blocks, ss_env_step_pool_blocks):

  1. the env step alone at 262,144 envs, M = n / 2 pool envs, K = 8 opponents: the block-rule step
     (ss_env_step_pool_blocks) with uniform blocks and with skewed blocks (one opponent holds half the pool) against the
     fixed-size step (ss_env_step_pool), per kernel with torch.profiler, each in a run of its own of `launches` launches;
  2. the whole pool tick (one ss_pool_rollout_frames call of `ticks` ticks, timed with CUDA events, best of `rounds`,
     the three trainers alternated) at 262,144 and 65,536 envs, M = n / 2, K = 8, of a trainer without a block table,
     one given the uniform table and one given the skewed table; a 1-frame learner against 1-frame opponents and a
     20-frame learner against 20-frame opponents;
  3. one set_pool_blocks (the restart kernel, the learner's history push and the opponents' new histories), host clock
     around the call and a device synchronise, best of `rounds`.

    python tools/pool_blocks_time.py [--ticks 32] [--rounds 3] [--launches 100] [--out DIR]

Setup: bf16 forwards, parameter noise 0.5 in groups of 128 rows, looking reward, random starts, the replay ring written in
place (default capacity, 8 ticks).  Prints the card's name, power limit and SM clocks read in the same run; --out DIR
writes the tables (r7_pool_blocks_step_262144.txt, r7_pool_blocks_time.txt)."""
import argparse
import ctypes
import os
import subprocess
import sys
import time

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


def skewed(M):
    """one opponent holds half the pool, the other K - 1 share the rest in even blocks"""
    rest = M // 2 // (K - 1) // 2 * 2
    return [M // 2] + [rest] * (K - 2) + [M - M // 2 - rest * (K - 2)]


def step_kernels(n, launches):
    """per-kernel device time of the three steps (torch.profiler), us per launch"""
    from torch.profiler import ProfilerActivity, profile
    M = n // 2
    L = 2 * n - M
    d = dict(device="cuda")
    g = torch.Generator(device="cuda").manual_seed(0)
    act = torch.rand(L, 2, generator=g, **d) * 2.4 - 1.2
    opp_act = torch.rand(M, 2, generator=g, **d) * 2.4 - 1.2
    obs, reward, done_rows = torch.empty(L, 12, **d), torch.empty(L, **d), torch.empty(L, dtype=torch.uint8, **d)
    opp_obs = torch.empty(M, 12, **d)
    done, winner = torch.empty(n, dtype=torch.uint8, **d), torch.empty(n, dtype=torch.uint8, **d)
    status, stats = torch.zeros(2 + 144, dtype=torch.int32, **d), torch.zeros(K, 8, dtype=torch.int64, **d)
    out, tables = [], []
    for name, blocks in (("ss_env_step_pool (PoolRows)", None), ("blocks, uniform", [M // K] * K), ("blocks, skewed", skewed(M))):
        env = SkillshotEnvs(n, random_positions=True, seed=1)
        table = None if blocks is None else (ctypes.c_int64 * K)(*blocks)

        def step(t):
            args = [env.state.data_ptr(), n, M, K, act.data_ptr(), opp_act.data_ptr(), obs.data_ptr(), None, reward.data_ptr(),
                    done_rows.data_ptr(), opp_obs.data_ptr(), done.data_ptr(), winner.data_ptr(), 1, 2000, 1, 5, t,
                    status.data_ptr(), 2, stats.data_ptr()]
            rc = lib.ss_env_step_pool(*(args + [None])) if table is None else lib.ss_env_step_pool_blocks(*(args + [table, None]))
            assert rc == 0
        for t in range(20):
            step(t)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for t in range(launches):
                step(100 + t)
            torch.cuda.synchronize()
        ev = [e for e in prof.key_averages() if "step_pp_obs_kernel" in e.key]
        assert len(ev) == 1, [e.key for e in prof.key_averages()]
        us = getattr(ev[0], "self_device_time_total", None) or ev[0].self_cuda_time_total
        out.append((name, blocks, us / ev[0].count))
        tables.append("== %s, blocks %s ==\n" % (name, blocks) +
                      prof.key_averages().table(sort_by="cuda_time_total", row_limit=6, max_name_column_width=70))
        del env
    return out, tables


def trainer(n, frames, blocks=None):
    kw = dict(seed=1, precision="bf16", param_noise_sd=0.5, noise_group=128, reward_mode="looking", tick_limit=2000, frames=frames)
    opp = [ActorCritic(seed=10 + k).actor if frames == 1 else FrameStackActor(8, frames=frames, seed=10 + k, device="cuda").params
           for k in range(K)]
    return SelfPlayTrainer(n, opponents=opp, pool_envs=n // 2, pool_blocks=blocks, **kw)


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
    base = steps[0][2]
    lines.append("env step alone, n=262144 M=131072 K=8, %d launches each, torch.profiler (launches not chained)" % args.launches)
    for name, blocks, us in steps:
        lines.append("%-30s %8.2f us  %6.3fx" % (name, us, us / base))
    print("\n".join(lines[1:]))
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "r7_pool_blocks_step_262144.txt"), "w") as f:
            f.write("\n".join(lines) + "\n\n" + "\n\n".join(tables) + "\n")

    rows = ["%-44s %10s %10s %10s %8s %8s %14s" % ("case", "no table", "uniform", "skewed", "uniform", "skewed", "set_pool_blocks")]
    print(rows[0])
    for n, frames in ((262144, 1), (65536, 1), (262144, 20), (65536, 20)):
        M = n // 2
        trs = [trainer(n, frames), trainer(n, frames, [M // K] * K), trainer(n, frames, skewed(M))]
        for tr in trs:
            tr.rollout(args.ticks)                   # warm-up: module loads, the ring's first pass
        best = [float("inf")] * 3
        for _ in range(args.rounds):
            for i, tr in enumerate(trs):
                best[i] = min(best[i], timed(tr, args.ticks))
        relayout = float("inf")
        tr = trs[2]
        for r in range(args.rounds + 1):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            tr.set_pool_blocks([M // K] * K if r % 2 == 0 else skewed(M))
            torch.cuda.synchronize()
            if r:                                    # (the first call is a warm-up)
                relayout = min(relayout, (time.perf_counter() - t0) * 1e3)
        row = "%-44s %7.1f us %7.1f us %7.1f us %7.3fx %7.3fx %11.2f ms" % (
            "n=%d M=%d K=8 x %d frames (learner %d)" % (n, M, frames, frames), best[0], best[1], best[2], best[1] / best[0],
            best[2] / best[0], relayout)
        print(row)
        rows.append(row)
        del trs, tr
        torch.cuda.empty_cache()
    if args.out:
        with open(os.path.join(args.out, "r7_pool_blocks_time.txt"), "w") as f:
            f.write(head + "\npool tick per trainer (one ss_pool_rollout_frames call of %d ticks, best of %d rounds, alternated); "
                    "ratios against the trainer without a block table; set_pool_blocks: host clock with a device synchronise, "
                    "best of %d\n" % (args.ticks, args.rounds, args.rounds) + "\n".join(rows) + "\n")


if __name__ == "__main__":
    main()
