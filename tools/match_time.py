"""Device time of one match tick (Match.advance: the policies' forwards + ss_env_step_match [+ history pushes]) against one
self-play rollout tick at the same env count (SelfPlayTrainer.rollout(store=False), param_noise_sd = 0: the same 2 n_envs
forward rows plus one env step, no noise draw), alternated in one process and timed with CUDA events after warm-up.

    python tools/match_time.py [--envs 65536 262144] [--ticks 64] [--rounds 3] [--profile DIR]

Cases per env count: 1-frame vs 1-frame actors (bf16), 20-frame vs 1-frame (bf16), and 1 vs 1 in float32 (65,536 only).
Also the wall time per tick of a whole Match.play() (one 128-byte summary read back per 64 ticks, stops when every game is
decided).  Prints the card's name and power limit.  --profile DIR writes torch.profiler per-kernel tables of 262,144-env
1 vs 1 match ticks and rollout ticks (a run of their own, after the timed ones).  The per-tick working set (env state,
observations, actions: 176 bytes per env, 46 MB at 262,144 envs) fits in the 126 MB L2 for the match and the rollout alike."""
import argparse
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from skillshot_learning_b200 import ActorCritic, Match, SelfPlayTrainer  # noqa: E402


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, nargs="+", default=[65536, 262144])
    ap.add_argument("--ticks", type=int, default=64)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--profile", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    print("card: %s" % card())
    K = args.ticks
    if (args.rounds + 1) * K > 2000:
        raise SystemExit("rounds x ticks must stay under the 2000-tick limit")
    actors = {f: ActorCritic(frames=f, seed=f).actor for f in (1, 20)}
    opp = ActorCritic(frames=1, seed=99).actor
    for n in args.envs:
        cases = [("1v1 bf16", 1, "bf16"), ("20v1 bf16", 20, "bf16")] + ([("1v1 f32", 1, "f32")] if n <= 65536 else [])
        for name, fa, prec in cases:
            m = Match(actors[fa], opp, n, precision=prec, seed=1)
            tr = SelfPlayTrainer(n, seed=1, precision=prec, param_noise_sd=0.0)
            m.advance(K)                                 # warm-up of every shape
            tr.rollout(K, store=False)
            torch.cuda.synchronize()
            tm, trl = [], []
            for _ in range(args.rounds):
                tm.append(timed(m.advance, K))
                trl.append(timed(lambda k: tr.rollout(k, store=False), K))
            t_m, t_r = min(tm), min(trl)
            print("envs %7d  %-9s  match tick %8.2f us (rounds: %s)  rollout tick %8.2f us (rounds: %s)  match / rollout %.3f" % (
                n, name, t_m, " ".join("%.2f" % x for x in tm), t_r, " ".join("%.2f" % x for x in trl), t_m / t_r))
            m2 = Match(actors[fa], opp, n, precision=prec, seed=2)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r = m2.play()
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
            print("envs %7d  %-9s  Match.play(): %d ticks, %.2f us per tick wall, score %.4f +- %.4f, draws %d, mean ticks decided %.1f" % (
                n, name, m2.ticks, wall / m2.ticks * 1e6, r["score"], r["score_stderr"], r["draws"], r["mean_ticks_decided"]))
            del m, m2, tr
            torch.cuda.empty_cache()
    if args.profile:
        from torch.profiler import ProfilerActivity, profile
        os.makedirs(args.profile, exist_ok=True)
        n = 262144
        m = Match(actors[1], opp, n, precision="bf16", seed=1)
        tr = SelfPlayTrainer(n, seed=1, precision="bf16", param_noise_sd=0.0)
        m.advance(K)
        tr.rollout(K, store=False)
        torch.cuda.synchronize()
        out = ["card: %s" % card()]
        for what, fn in (("match ticks (1 vs 1, bf16)", m.advance), ("rollout ticks (store=False, no noise, bf16)",
                                                                      lambda k: tr.rollout(k, store=False))):
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                fn(K)
                torch.cuda.synchronize()
            table = prof.key_averages().table(sort_by="cuda_time_total", row_limit=12)
            out.append("%d %s at %d envs\n%s" % (K, what, n, table))
        text = "\n".join(out)
        with open(os.path.join(args.profile, "match_kernels_262144.txt"), "w") as f:
            f.write(text + "\n")
        print(text)


if __name__ == "__main__":
    main()
