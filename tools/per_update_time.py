"""Time of the prioritized draw and of the prioritized update against the uniform ones, alternated in one process with
CUDA events after warm-up (best of --rounds rounds of --reps calls).

    python tools/per_update_time.py [--rows 65536] [--reps 20] [--rounds 3]

Rings filled by 8 rollout ticks of rows / 2 envs (a full ring of 8 x rows rows, terminal reward), bf16.  For n = 1 and 3:
(a) the sampler alone on the 12-input ring and on the 20-frame ring (uniform: ss_replay_sample / ss_replay_sample_nstep;
prioritized: ss_replay_sample_prioritized, its three launches), as the kernels' device time from torch.profiler; (b) update()
of the 12-input networks (one ss_ddpg_update call) and of the 20-frame networks (separate steps), prioritized against
uniform.  The prioritized trainers run a few updates first, so that their leaves are no longer all equal.  Prints the
card's name, power limit and maximum SM clock first."""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from skillshot_learning_b200 import SelfPlayTrainer  # noqa: E402

NS = (1, 3)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.SubprocessError):
        q = torch.cuda.get_device_name(0) + ", power limit and clock unknown"
    return q


def timed(fns, reps, rounds):
    """name -> best of `rounds` mean ms per call of fns[name], the names alternated within each round"""
    for f in fns.values():                                   # warm-up of every shape
        for _ in range(4):
            f()
    torch.cuda.synchronize()
    best = {k: float("inf") for k in fns}
    for _ in range(rounds):
        for k, f in fns.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                f()
            e1.record()
            e1.synchronize()
            best[k] = min(best[k], e0.elapsed_time(e1) / reps)
    return best


def kernel_us(f, reps):
    """mean device time (us) of the sampling kernels (replay_sample*, priority_scan / priority_blocks) of `reps` calls of f"""
    from torch.profiler import ProfilerActivity, profile
    for _ in range(3):
        f()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            f()
        torch.cuda.synchronize()
    tot = 0.0
    for e in prof.key_averages():
        if "replay_sample" in e.key or "priority_scan" in e.key or "priority_blocks" in e.key:
            tot += getattr(e, "device_time_total", None) or e.cuda_time_total
    return tot / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=65536)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    print("card: %s" % card())
    rows = args.rows
    for frames in (1, 20):
        label = "%s networks, bf16, %d rows" % ("12-input" if frames == 1 else "20-frame", rows)
        tr = {}
        for n in NS:
            for pri in (False, True):
                t = SelfPlayTrainer(rows // 2, device="cuda:0", seed=1, batch_size=rows, gamma=0.99, tau=0.005,
                                    reward_mode="terminal", tick_limit=200, precision="bf16", frames=frames, update_precision="bf16",
                                    replay_capacity=8 * rows, n_step=n, prioritized_replay=pri)
                t.rollout(8)
                if pri:
                    for _ in range(4):
                        t.update()
                tr[n, pri] = t
        ring = tr[1, True].replay
        print("%s: ring of %d rows, %d with a hit; leaves min %.3g max %.3g, priority_max %.3g" % (
            label, ring.size, int(ring.done.sum()), float(ring.priority.min()), float(ring.priority.max()),
            float(ring.priority_max)))
        fns = {}
        for n in NS:
            for pri in (False, True):
                rg = tr[n, pri].replay
                kw = dict(n_step=n, gamma=0.99, beta=0.4 if pri else None)
                o = rg.sample(rows, **kw)
                fns["sampler n = %d %s" % (n, "prioritized" if pri else "uniform")] = (lambda rg=rg, o=o, kw=kw: rg.sample(rows, out=o, **kw))
        ks = {k: kernel_us(f, args.reps) for k, f in fns.items()}
        for n in NS:
            u, p = ks["sampler n = %d uniform" % n], ks["sampler n = %d prioritized" % n]
            print("%-36s kernels, sampler n = %d: uniform %8.2f us, prioritized %8.2f us  (%.2fx)" % (label, n, u, p, p / u))
        best = timed({"update() n = %d %s" % (n, "prioritized" if pri else "uniform"): tr[n, pri].update
                      for n in NS for pri in (False, True)}, args.reps, args.rounds)
        for n in NS:
            u, p = best["update() n = %d uniform" % n], best["update() n = %d prioritized" % n]
            print("%-36s update(), n = %d: uniform %.4f ms, prioritized %.4f ms  (%.3fx)" % (label, n, u, p, p / u))
        del tr, ring, fns
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
