"""Time of n-step sampling and of the update on n-step rows against one-step rows, alternated in one process with CUDA
events after warm-up (best of --rounds rounds of --reps calls).

    python tools/nstep_update_time.py [--rows 65536] [--reps 20] [--rounds 3]

Rings filled by 8 rollout ticks of rows / 2 envs (a full ring of 8 x rows rows, terminal reward), bf16.  For n = 1, 3, 5:
(a) the sampler alone on the 12-input ring and on the 20-frame ring (n = 1: ss_replay_sample; n > 1: ss_replay_sample_nstep;
also ss_replay_sample_nstep at n = 1, the same rows), as calls timed with CUDA events (bound by the host at these sizes) and
as the kernel's device time from torch.profiler; (b) update() of the 12-input networks (one ss_ddpg_update call) and of
the 20-frame networks (separate steps).  Prints the card's name, power limit and maximum SM clock first."""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from skillshot_learning_b200 import SelfPlayTrainer  # noqa: E402

NS = (1, 3, 5)


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
    """mean device time (us) of the replay_sample* kernels of `reps` calls of f, from torch.profiler"""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            f()
        torch.cuda.synchronize()
    tot = 0.0
    for e in prof.key_averages():
        if "replay_sample" in e.key:
            tot += getattr(e, "device_time_total", None) or e.cuda_time_total
    return tot / reps


def report(label, best, ref):
    for k, v in best.items():
        print("%-40s %-30s %8.4f ms  %.3fx of %s" % (label, k, v, v / best[ref], ref))


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
            t = SelfPlayTrainer(rows // 2, device="cuda:0", seed=1, batch_size=rows, gamma=0.99, tau=0.005, reward_mode="terminal",
                                tick_limit=200, precision="bf16", frames=frames, update_precision="bf16",
                                replay_capacity=8 * rows, n_step=n)
            t.rollout(8)
            tr[n] = t
        ring = tr[3].replay
        print("%s: ring of %d rows, %d with a hit; eligible rows n = 3: %d, n = 5: %d" % (
            label, ring.size, int(ring.done.sum()), sum(l for _, l in ring.eligible_runs(3)),
            sum(l for _, l in ring.eligible_runs(5))))
        outs = {}
        fns = {"sampler n = 1 (ss_replay_sample)": lambda: ring.sample(rows, out=outs.get(1))}
        import ctypes
        from skillshot_learning_b200 import _lib
        o1 = ring.sample(rows, n_step=3, gamma=0.99)
        table = (ctypes.c_int64 * 2)(0, ring.size)

        def nstep_one():
            _lib.check(_lib.lib.ss_replay_sample_nstep(
                ring.obs.data_ptr(), ring.act.data_ptr(), ring.reward.data_ptr(), ring.next_obs.data_ptr(), ring.done.data_ptr(),
                ring.capacity, ring.frames, ring.tick_rows, 1, 0.99, table, 1, ring.seed, ring.counter, rows,
                *[o1[k].data_ptr() for k in ("obs", "act", "reward", "next_obs", "done", "indices", "steps")],
                torch.cuda.current_stream().cuda_stream), "ss_replay_sample_nstep")
        fns["sampler n = 1 (ss_replay_sample_nstep)"] = nstep_one
        for n in NS[1:]:
            o = ring.sample(rows, n_step=n, gamma=0.99)
            fns["sampler n = %d" % n] = (lambda n=n, o=o: ring.sample(rows, out=o, n_step=n, gamma=0.99))
        outs[1] = ring.sample(rows)
        best = timed(fns, args.reps, args.rounds)
        report(label + ", sampler (host-bound)", best, "sampler n = 1 (ss_replay_sample)")
        best = {k: kernel_us(f, args.reps) for k, f in fns.items()}
        for k, v in best.items():
            print("%-40s %-40s %8.2f us  %.3fx" % (label + ", kernel", k, v, v / best["sampler n = 1 (ss_replay_sample)"]))
        best = timed({"update() n = %d" % n: tr[n].update for n in NS}, args.reps, args.rounds)
        report(label, best, "update() n = 1")
        del tr, ring, fns, outs, o1
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
