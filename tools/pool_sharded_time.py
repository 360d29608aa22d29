"""Weak scaling of training against a pool of frozen opponents on several GPUs (SelfPlayTrainer(opponents=...,
process_group=True), DESIGN.md section 6.13).  Every rank holds the same per-GPU problem; the time of one training
iteration -- rollout(4) then update() -- is measured with CUDA events, best of `rounds` rounds of `iters` iterations,
and the maximum over the ranks is reported, for each collective ("nccl", "peer"; one GPU: no group).  Two cases per GPU:

  a. config 5: 65,536 envs, M = 32,768 pool envs, 8 twenty-frame opponents and a 20-frame learner, bf16 forward and
     update, a speed sweep U(0.5, 2) x the reference constants, parameter noise 0.5 in groups of 128, batch 65,536,
     gamma 0.99, tau 0.005;
  b. a 1-frame pool: 262,144 envs, M = 131,072, K = 8, bf16, the same noise, batch, gamma and tau.

Also the host time, with a device synchronise, of one pool_progress() and one rebalance_pool() (median of 5, maximum
over the ranks).

    python tools/pool_sharded_time.py [--out DIR]                                   # N = 1, no group
    python -m torch.distributed.run --nproc-per-node N tools/pool_sharded_time.py [--out DIR]

Prints the card's name and power limit read in the same run.  --out DIR appends the table to
DIR/r9_pool_sharded_time.txt and writes DIR/pool_sharded_N{N}.json; the weak-scaling efficiency t_1 / t_N is printed when
DIR/pool_sharded_N1.json (the N = 1 run) is there."""
import argparse
import json
import os
import subprocess
import sys
import time

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from skillshot_learning_b200 import SelfPlayTrainer  # noqa: E402
from skillshot_learning_b200._lib import lib  # noqa: E402

K = 8
CASES = {
    "a: config 5, 65536 envs, M 32768, 8 x 20-frame opponents, 20-frame learner, speeds":
        dict(n=65536, M=32768, frames=20, speeds=True),
    "b: 1-frame pool, 262144 envs, M 131072, 8 opponents": dict(n=262144, M=131072, frames=1, speeds=False),
}


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name(0) + ", power limit unknown"


def sweep(n, seed, dev):
    """bench.py's configs[4] speeds: each constant U(0.5, 2) times the reference's, the cooldown rounded, at least 1"""
    g = torch.Generator(device=dev).manual_seed(seed)
    scale = lambda: 0.5 + 1.5 * torch.rand(n, device=dev, generator=g)
    return 3.0 * scale(), 0.25 * scale(), 5.0 * scale(), (15.0 * scale()).round().clamp(min=1)


def trainer(case, rank, dev, group, collective):
    c = CASES[case]
    f = c["frames"]
    g = torch.Generator().manual_seed(10)
    opp = [torch.randn(int(lib.ss_actor_frames_params(f)), generator=g) * 0.05 for _ in range(K)]
    tr = SelfPlayTrainer(c["n"], device=dev, seed=1 + rank, opponents=opp, pool_envs=c["M"], frames=f, precision="bf16",
                         update_precision="bf16", param_noise_sd=0.5, noise_group=128, batch_size=65536, gamma=0.99, tau=0.005,
                         reward_mode="looking", tick_limit=2000, process_group=group, collective=collective)
    if c["speeds"]:
        tr.envs.set_speeds(*sweep(c["n"], 3 + rank, dev))
    return tr


def max_over_ranks(x, world):
    if world == 1:
        return x
    got = [None] * world
    dist.all_gather_object(got, x)
    return max(got)


def barrier(world):
    if world > 1:
        dist.barrier()


def iteration_ms(tr, iters, rounds, world):
    for _ in range(4):                       # warm-up: module loads, the ring's first pass, the update's buffers
        tr.rollout(4)
        tr.update()
    torch.cuda.synchronize()
    best = float("inf")
    for _ in range(rounds):
        barrier(world)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            tr.rollout(4)
            tr.update()
        b.record()
        b.synchronize()
        best = min(best, a.elapsed_time(b) / iters)
    return max_over_ranks(best, world)


def host_ms(fn, world, reps=5):
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        barrier(world)
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return max_over_ranks(sorted(ts)[reps // 2], world)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=16)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank, local = int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        group = True
    head = card()
    lines = ["N = %d GPU(s); one iteration = rollout(4) + update(), best of %d rounds of %d iterations, maximum over ranks"
             % (world, args.rounds, args.iters), head]
    base = None
    if args.out and os.path.exists(os.path.join(args.out, "pool_sharded_N1.json")):
        base = json.load(open(os.path.join(args.out, "pool_sharded_N1.json")))
    lines.append("%-82s %-6s %12s %10s %16s %16s" % ("case", "coll.", "iteration", "t1 / tN", "pool_progress", "rebalance_pool"))
    results = {}
    for case in CASES:
        for collective in (("nccl", "peer") if world > 1 else ("none",)):
            tr = trainer(case, rank, dev, group, "nccl" if collective == "none" else collective)
            ms = iteration_ms(tr, args.iters, args.rounds, world)
            prog = host_ms(lambda: tr.pool_progress(), world)
            reb = host_ms(lambda: tr.rebalance_pool(), world)
            tr.check_exchange()
            tr.envs.check_status()
            if tr.networks.peer is not None:
                tr.networks.peer.close()
            del tr
            torch.cuda.empty_cache()
            key = "%s | %s" % (case, collective)
            results[key] = dict(iteration_ms=ms, pool_progress_ms=prog, rebalance_pool_ms=reb)
            t1 = None if base is None else base.get("%s | none" % case, {}).get("iteration_ms")
            eff = "%10.3f" % (t1 / ms) if t1 else "%10s" % "-"
            lines.append("%-82s %-6s %9.3f ms %s %13.3f ms %13.3f ms" % (case, collective, ms, eff, prog, reb))
            if rank == 0:
                print(lines[-1], flush=True)
    if rank == 0:
        print("\n".join(lines[:2]))
        if args.out:
            os.makedirs(args.out, exist_ok=True)
            with open(os.path.join(args.out, "pool_sharded_N%d.json" % world), "w") as f:
                json.dump(dict(card=head, world=world, results=results), f, indent=1)
            with open(os.path.join(args.out, "r9_pool_sharded_time.txt"), "a") as f:
                f.write("\n".join(lines) + "\n\n")
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
