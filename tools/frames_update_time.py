"""Time of one update of the 20-frame networks (TD target + critic step + actor step), float32 kernels against the
tensor-core kernels, alternated in one process with CUDA events after warm-up.

    python tools/frames_update_time.py [--rows 65536 262144] [--reps 20] [--rounds 3] [--profile DIR]

Prints the card's name and power limit, the FLOPs of an update computed from the layer shapes, the time per update,
rows/s and the share of the dense bf16 peak (2,250 TFLOP/s, B200 data sheet, 1000 W).  --profile DIR also writes a
torch.profiler per-kernel table of the bf16 update (a run of its own, after the timed one)."""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from skillshot_learning_b200 import ActorCritic  # noqa: E402

BF16_PEAK = 2250e12


def flops_per_row(frames):
    """Multiply-adds x 2 of the dense layers the update runs per row."""
    l1, l2c, l2a = 12 * frames * 256, 258 * 128, 256 * 128
    fwd_a, fwd_c = l1 + l2a + 128 * 2, l1 + l2c + 128
    target = fwd_a + fwd_c                                   # a' = actor'(s'), q' = critic'(s', a')
    critic = fwd_c + (128 + l2c + 256 * 128) + l1            # forward, dW3 + dW2 + dx2, dW1
    actor = fwd_a + fwd_c + (256 + l2a + 256 * 128) + l1     # a, q and -dQ/da, backward through the actor
    return 2 * (target + critic + actor)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.SubprocessError):
        q = torch.cuda.get_device_name(0) + ", power limit unknown"
    return q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, nargs="+", default=[65536, 262144])
    ap.add_argument("--frames", type=int, default=20)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--profile", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    F = args.frames
    print("card: %s" % card())
    print("frames %d: %.3f MFLOP per row and update" % (F, flops_per_row(F) / 1e6))
    g = torch.Generator(device="cuda").manual_seed(0)
    for n in args.rows:
        s = torch.rand((n, 12 * F), device="cuda", generator=g)
        s2 = torch.rand((n, 12 * F), device="cuda", generator=g)
        a = torch.rand((n, 2), device="cuda", generator=g) * 2 - 1
        r = -torch.rand(n, device="cuda", generator=g)
        nets = {p: ActorCritic(device="cuda:0", seed=1, frames=F, gamma=0.9, tau=0.05, update_precision=p) for p in ("f32", "bf16")}
        theta, phi = nets["f32"].actor.clone(), nets["f32"].critic.clone()

        def update(ac):
            y = ac.td_targets(r, s2)
            ac.critic_step(s, a, y)
            ac.actor_step(s)

        times = {p: [] for p in nets}
        for p, ac in nets.items():                           # warm-up of every shape
            ac.set_weights(theta, phi)
            for _ in range(3):
                update(ac)
        torch.cuda.synchronize()
        for _ in range(args.rounds):
            for p, ac in nets.items():
                ac.set_weights(theta, phi)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.reps):
                    update(ac)
                e1.record()
                e1.synchronize()
                times[p].append(e0.elapsed_time(e1) / args.reps)
        for p in nets:
            t = min(times[p]) * 1e-3
            fl = flops_per_row(F) * n
            print("rows %7d  %-4s  %8.3f ms/update (rounds: %s)  %.3g rows/s  %.1f TFLOP/s  %.4f of bf16 peak" % (
                n, p, t * 1e3, " ".join("%.3f" % x for x in times[p]), n / t, fl / t / 1e12, fl / t / BF16_PEAK))
        print("rows %7d  speed-up bf16 / f32: %.2fx" % (n, min(times["f32"]) / min(times["bf16"])))
        if args.profile:
            from torch.profiler import ProfilerActivity, profile
            os.makedirs(args.profile, exist_ok=True)
            ac = nets["bf16"]
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(args.reps):
                    update(ac)
                torch.cuda.synchronize()
            table = prof.key_averages().table(sort_by="cuda_time_total", row_limit=20)
            with open(os.path.join(args.profile, "frames_update_kernels_%d.txt" % n), "w") as f:
                f.write("card: %s\n%d updates of %d rows, bf16\n%s\n" % (card(), args.reps, n, table))
            print(table)


if __name__ == "__main__":
    main()
