"""Device time of one rollout tick of a 20-frame learner that plays part of its envs against a pool of frozen opponents
(SelfPlayTrainer(frames=20, opponents=...).rollout: one ss_pool_rollout_frames call) against one tick of the frame-stacked
self-play trainer at the same env count (SelfPlayTrainer(frames=20).rollout: noise vectors, forward, env step, two history
pushes, the ordered rows and the ring push, per tick from Python), alternated in one process and timed with CUDA events.

    python tools/pool_frames_rollout_time.py [--ticks 16] [--rounds 3] [--profile DIR]

Setup of both: bf16 forwards, 20-frame learner, parameter noise 0.5 in groups of 128 rows, looking reward, random starts,
the replay ring written in place (default capacity, 8 ticks).  Cases at 65,536 envs (the 131,072 player rows of the
20-frame configuration): M = n / 2 pool envs against K = 8 twenty-frame opponents, against K = 8 mixed opponents (four with
1 frame, four with 20), and M = 0 (the pool path with no pool envs); and M = n / 2, K = 8 twenty-frame opponents at
262,144 envs.  Each round times one call of `ticks` ticks per trainer after a warm-up call; a case reports the best of its
rounds, per tick.  Prints the card's name, power limit and SM clocks read in the same run.  --profile DIR also writes the
files committed under profiles/: the timed table (r6_pool_frames_time.txt), torch.profiler per-kernel tables of 4 ticks of
the M = n / 2, K = 8 twenty-frame pool trainer and of the self-play trainer at 65,536 envs
(r6_pool_frames_kernels_{pool,selfplay}_65536.txt, a run of its own after the timed ones with the launches not chained:
ss_set_dependent_launch(0)), and the history step's bytes and rates, ss_obs_stack_push_pool against the four launches it
replaces (r6_pool_frames_push_65536.txt)."""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from skillshot_learning_b200 import SelfPlayTrainer  # noqa: E402
from skillshot_learning_b200._lib import lib  # noqa: E402

F = 20
HBM_BYTES_PER_S = 7.7e12         # HGX B200 data sheet, one GPU


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


def actor(frames, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(int(lib.ss_actor_frames_params(frames)), generator=g) * 0.05


def trainer(n, M=None, opp_frames=()):
    kw = dict(seed=1, precision="bf16", param_noise_sd=0.5, noise_group=128, reward_mode="looking", tick_limit=2000, frames=F)
    if opp_frames:
        kw.update(opponents=[actor(f, 10 + k) for k, f in enumerate(opp_frames)], pool_envs=M)
    return SelfPlayTrainer(n, **kw)


def push_bytes(frames):
    """HBM bytes per learner row of one history step without a restart: (fused, the composition it replaces)"""
    w = 48 * frames
    fused = 48 + 48 * (frames - 1) + 48 + 28 + 2 * w           # obs, the other slots, float32 slot, fp16 slot + {1, 1}, two rows
    comp = ((48 + 28) + (48 + 48) + (w + w) +                 # push_tc, push, ordered (reads every slot, writes the row)
            (2 * w + 2 * w + 2 * (8 + 4 + 1)))                # ring push: reads both rows, writes both, act / reward / done
    return fused, comp


def profile_case(name, tr, out_dir, n):
    from torch.profiler import ProfilerActivity, profile
    tr.rollout(8)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        tr.rollout(4)
        torch.cuda.synchronize()
    avg = prof.key_averages()
    with open(os.path.join(out_dir, "r6_pool_frames_kernels_%s_%d.txt" % (name, n)), "w") as f:
        f.write(card() + "\n4 rollout ticks, %d envs, bf16, 20-frame learner, launches not chained\n" % n)
        f.write(avg.table(sort_by="cuda_time_total", row_limit=25, max_name_column_width=70))
    times = {}
    for e in avg:
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        times[e.key] = (t, e.count)
    return times


def kernel_us(times, needle):
    hits = [(t, c) for k, (t, c) in times.items() if needle in k]
    return sum(t for t, _ in hits) / max(1, sum(c for _, c in hits)) if hits else float("nan")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ticks", type=int, default=16)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--profile", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)
    say(card())
    cases = [(65536, 32768, [F] * 8, "K=8 x 20 frames"), (65536, 32768, [1] * 4 + [F] * 4, "K=8 mixed 4 x 1, 4 x 20"),
             (65536, 0, [F], "no pool envs"), (262144, 131072, [F] * 8, "K=8 x 20 frames")]
    say("%-46s %12s %14s %7s" % ("case", "pool tick", "self-play tick", "ratio"))
    for n, M, opp, label in cases:
        pool, selfplay = trainer(n, M, opp), trainer(n)
        for tr in (pool, selfplay):
            tr.rollout(args.ticks)                   # warm-up: module loads, the ring's first pass
        best_p = best_s = float("inf")
        for _ in range(args.rounds):
            best_p = min(best_p, timed(pool, args.ticks))
            best_s = min(best_s, timed(selfplay, args.ticks))
        say("%-46s %9.1f us %11.1f us %6.3fx" % ("n=%d M=%d %s" % (n, M, label), best_p, best_s, best_p / best_s))
        del pool, selfplay
        torch.cuda.empty_cache()
    if args.profile:
        os.makedirs(args.profile, exist_ok=True)
        with open(os.path.join(args.profile, "r6_pool_frames_time.txt"), "w") as f:
            f.write("\n".join(lines) + "\n")
        n, M = 65536, 32768
        lib.ss_set_dependent_launch(0)
        tp = profile_case("pool", trainer(n, M, [F] * 8), args.profile, n)
        torch.cuda.empty_cache()
        ts = profile_case("selfplay", trainer(n), args.profile, n)
        lib.ss_set_dependent_launch(1)
        fused_b, comp_b = push_bytes(F)
        L_pool, L_self = 2 * n - M, 2 * n
        fused_us = kernel_us(tp, "obs_stack_push_pool_kernel")
        parts = [(k, kernel_us(ts, k)) for k in ("obs_stack_push_tc_kernel", "obs_stack_push_kernel", "obs_stack_ordered_kernel",
                                                 "replay_push_kernel")]
        comp_us = sum(t for _, t in parts)
        with open(os.path.join(args.profile, "r6_pool_frames_push_%d.txt" % n), "w") as f:
            f.write(card() + "\nthe learner's history step per tick, %d envs, 20 frames, bf16, launches not chained\n" % n)
            f.write("ss_obs_stack_push_pool (pool, %d rows): %.1f us, %d B/row, %.2f TB/s (%.0f %% of 7.7 TB/s)\n" % (
                L_pool, fused_us, fused_b, L_pool * fused_b / fused_us / 1e6, 100 * L_pool * fused_b / fused_us / 1e6 / 7.7))
            f.write("composition (self-play, %d rows): %.1f us, %d B/row, %.2f TB/s (%.0f %% of 7.7 TB/s)\n" % (
                L_self, comp_us, comp_b, L_self * comp_b / comp_us / 1e6, 100 * L_self * comp_b / comp_us / 1e6 / 7.7))
            for k, t in parts:
                f.write("  %-28s %.1f us\n" % (k, t))
            f.write("per row: fused %.3f ns, composition %.3f ns\n" % (1e3 * fused_us / L_pool, 1e3 * comp_us / L_self))
        print(open(os.path.join(args.profile, "r6_pool_frames_push_%d.txt" % n)).read())


if __name__ == "__main__":
    main()
