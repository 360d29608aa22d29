"""Time of one TD3 update (twin critics, policy delay 2, target noise 0.2 clipped at 0.5) against one DDPG update of the same
trainer configuration, alternated in one process with CUDA events after warm-up (best of --rounds rounds of --reps updates;
a TD3 figure is the mean over its delay cycle, half of its updates run the actor step).

    python tools/td3_update_time.py [--rows 65536] [--reps 20] [--rounds 3]

Cases: (a) the 12-input networks on the tensor cores, DDPG through update() (one ss_ddpg_update call) and through
update_stepwise(), TD3 through update() (which runs the separate steps); (b) the 20-frame networks on the tensor cores.
Also the TD target alone, ss_td3_targets* (two critics, smoothing) against ss_ddpg_targets*.  Prints the card's name, power
limit and maximum SM clock first."""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from skillshot_learning_b200 import SelfPlayTrainer  # noqa: E402

TD3 = dict(twin_critics=True, policy_delay=2, target_noise=0.2, target_noise_clip=0.5)


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


def trainers(rows, frames):
    kw = dict(device="cuda:0", seed=1, batch_size=rows, gamma=0.99, tau=0.005, reward_mode="terminal", tick_limit=200,
              precision="bf16", frames=frames, update_precision="bf16")
    n_envs = rows // 2
    out = {}
    for name, extra in (("ddpg", {}), ("td3", TD3)):
        t = SelfPlayTrainer(n_envs, replay_capacity=8 * rows, **kw, **extra)
        t.rollout(8)                                         # a full ring: 8 ticks of 2 n_envs = rows rows
        out[name] = t
    return out


def report(label, best, ref):
    for k, v in best.items():
        print("%-44s %-22s %8.3f ms  %.3fx of %s" % (label, k, v, v / best[ref], ref))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=65536)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    print("card: %s" % card())
    n = args.rows
    for frames, label in ((1, "(a) 12-input networks, bf16, %d rows" % n), (20, "(b) 20-frame networks, bf16, %d rows" % n)):
        tr = trainers(n, frames)
        fns = {"DDPG update_stepwise()": tr["ddpg"].update_stepwise, "TD3 update()": tr["td3"].update}
        if frames == 1:
            fns = {"DDPG update()": tr["ddpg"].update, **fns}
        best = timed(fns, args.reps, args.rounds)
        report(label, best, "DDPG update()" if frames == 1 else "DDPG update_stepwise()")
        b = tr["td3"].replay.sample(n)
        nets = {k: tr[k].networks for k in tr}
        best = timed({"ss_ddpg_targets%s" % ("_tc" if frames == 1 else "_frames_tc"):
                      lambda: nets["ddpg"].td_targets(b["reward"], b["next_obs"], b["done"]),
                      "ss_td3_targets%s" % ("_tc" if frames == 1 else "_frames_tc"):
                      lambda: nets["td3"].td_targets(b["reward"], b["next_obs"], b["done"])}, args.reps, args.rounds)
        report(label + ", target alone", best, next(iter(best)))
        del tr, nets, b
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
