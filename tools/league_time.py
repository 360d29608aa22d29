"""Device time of one league tick (League.advance: the segments' forwards + ss_env_step_seated [+ history pushes]) against
one two-policy Match tick at the same game count, alternated in one process and timed with CUDA events after warm-up.

    python tools/league_time.py [--ticks 32] [--rounds 3] [--profile DIR]

Cases (bf16):
  (a) 16 one-frame policies, round robin, 2,048 games per pair (245,760 games) -- against a 1 vs 1 Match of 245,760 games;
      the ratio is the cost of generality
  (b) gauntlet of 1 vs 8, 32,768 games per pair (262,144 games) -- against a Match of 262,144 games
  (c) 64 one-frame policies, round robin, 128 games per pair (258,048 games: many short segments) -- against a Match
  (d) four policies, one of them with 20 frames, round robin, 16,384 games per pair (98,304 games) -- against a 20 vs 1
      Match of the same count
Also the wall time of a whole League.play() per case (one [P][P][8] summary read back per 64 ticks, stops when every
game is decided).  Prints the card's name and power limit.  --profile DIR writes torch.profiler per-kernel tables of case
(a) and of its Match (the segment forward beside the grouped forward, the seated step beside the match step), a run of
its own after the timed ones.  Working set per tick: 176 bytes per env (state, observations, actions), 43 MB at 245,760
envs, inside the 126 MB L2 for the league and the match alike."""
import argparse
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from skillshot_learning_b200 import ActorCritic, League, Match  # noqa: E402
from skillshot_learning_b200.league import gauntlet, round_robin  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.SubprocessError):
        q = torch.cuda.get_device_name(0) + ", power limit unknown"
    return q


def timed(fn, n_ticks):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn(n_ticks)
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / n_ticks * 1e3          # us per tick


def cases():
    a = lambda f, s: ActorCritic(frames=f, seed=s).actor      # noqa: E731
    return [
        ("(a) 16 x 1f round robin, 2048/pair", [a(1, 10 + k) for k in range(16)], None, 2048, (1, 1)),
        ("(b) gauntlet 1 vs 8, 32768/pair", [a(1, 30 + k) for k in range(9)], "gauntlet", 32768, (1, 1)),
        ("(c) 64 x 1f round robin, 128/pair", [a(1, 100 + k) for k in range(64)], None, 128, (1, 1)),
        ("(d) 4 policies incl. one 20f, 16384/pair", [a(1, 200), a(20, 201), a(1, 202), a(1, 203)], None, 16384, (20, 1)),
    ]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ticks", type=int, default=32)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--profile", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    print("card: %s" % card())
    K = args.ticks
    if (args.rounds + 1) * K > 2000:
        raise SystemExit("rounds x ticks must stay under the 2000-tick limit")
    for name, actors, sched, g, mf in cases():
        pairs = gauntlet(len(actors)) if sched == "gauntlet" else round_robin(len(actors))
        n = len(pairs) * g
        lg = League(actors, g, pairs=pairs, seed=1)
        m = Match(ActorCritic(frames=mf[0], seed=7).actor, ActorCritic(frames=mf[1], seed=8).actor, n, seed=1)
        lg.advance(K)                                    # warm-up of every shape
        m.advance(K)
        torch.cuda.synchronize()
        tl, tm = [], []
        for _ in range(args.rounds):
            tl.append(timed(lg.advance, K))
            tm.append(timed(m.advance, K))
        t_l, t_m = min(tl), min(tm)
        print("%-42s games %7d  league tick %8.2f us (rounds: %s)  match tick (%dv%d) %8.2f us (rounds: %s)  league / match %.3f" % (
            name, n, t_l, " ".join("%.2f" % x for x in tl), mf[0], mf[1], t_m, " ".join("%.2f" % x for x in tm), t_l / t_m))
        del lg, m
        lg2 = League(actors, g, pairs=pairs, seed=2)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = lg2.play()
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        print("%-42s League.play(): %d ticks, %.3f s wall (%.2f us per tick), seat-1 score %.4f +- %.4f, rating spread %.1f, "
              "median rating stderr %.1f" % (name, lg2.ticks, wall, wall / lg2.ticks * 1e6, r["seat1_score"], r["seat1_score_stderr"],
                                             float(r["ratings"].max() - r["ratings"].min()), float(sorted(r["rating_stderr"])[len(actors) // 2])))
        del lg2
        torch.cuda.empty_cache()
    if args.profile:
        from torch.profiler import ProfilerActivity, profile
        os.makedirs(args.profile, exist_ok=True)
        name, actors, _, g, _ = cases()[0]
        n = len(round_robin(len(actors))) * g
        lg = League(actors, g, seed=1)
        m = Match(ActorCritic(frames=1, seed=7).actor, ActorCritic(frames=1, seed=8).actor, n, seed=1)
        lg.advance(K)
        m.advance(K)
        torch.cuda.synchronize()
        out = ["card: %s" % card()]
        for what, fn in (("league ticks " + name, lg.advance), ("match ticks (1 vs 1, bf16)", m.advance)):
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                fn(K)
                torch.cuda.synchronize()
            table = prof.key_averages().table(sort_by="cuda_time_total", row_limit=12)
            out.append("%d %s at %d games\n%s" % (K, what, n, table))
        text = "\n".join(out)
        with open(os.path.join(args.profile, "league_kernels_245760.txt"), "w") as f:
            f.write(text + "\n")
        print(text)


if __name__ == "__main__":
    main()
