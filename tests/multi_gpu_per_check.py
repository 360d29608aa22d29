"""Run under torchrun with 2 GPUs (tests/test_gpu_multi_per.py launches it): prioritized updates sharded over the ranks.

With each collective (NCCL all-reduce, peer exchange), sharded trainers with prioritized replay -- self-play with the
12-input networks in bf16 (single-call update with the peer exchange), a pool with n_step = 3 and breaks, and TD3 with the
20-frame networks -- hold identical parameters, targets and Adam moments on every rank after rollout + update iterations
(torch.equal), while each rank draws from, weights by and writes the leaves of its own ring."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import learner_oracle as lo  # noqa: E402
from skillshot_learning_b200 import SelfPlayTrainer  # noqa: E402

CASES = {
    "self-play, 12-input, bf16": dict(precision="bf16"),
    "pool with breaks, n = 3": dict(precision="bf16", pool=True, n_step=3),
    "TD3, 20-frame": dict(frames=20, twin_critics=True, policy_delay=2, target_noise=0.2),
}


def _gather(t):
    out = [torch.empty_like(t) for _ in range(dist.get_world_size())]
    dist.all_gather(out, t.contiguous())
    return out


def check(case, collective, rank, dev, say):
    kw = dict(CASES[case])
    rows = 1024                                               # learner rows per tick; a ring of 16 ticks keeps the break
    if kw.pop("pool", False):
        rng = np.random.default_rng(1)                        # the same pool on every rank
        kw.update(opponents=[lo.init_actor(rng), lo.init_actor(rng)], pool_envs=256)
        rows = 768
    tr = SelfPlayTrainer(512, device=dev, seed=40 + rank, batch_size=1024, gamma=0.99, tau=0.05, tick_limit=30, process_group=True,
                         collective=collective, replay_capacity=16 * rows, prioritized_replay=True, **kw)
    tr.rollout(4)
    tr.rollout(1, store=False)
    if tr.opponents is not None:
        tr.set_pool_blocks([128, 128])
    for _ in range(5):
        tr.rollout(2)
        tr.update()
    torch.cuda.synchronize(dev)
    assert tr.replay.prioritized and float(tr.replay.priority_max) > 0, case
    net = tr.networks
    for k in ("params", "target", "adam_m", "adam_v"):
        got = _gather(getattr(net, k))
        assert all(torch.equal(got[0], x) for x in got[1:]), (case, collective, k)
    if net.peer is not None:
        tr.check_exchange()
        net.peer.close()
    say("%s, %s: identical parameters, targets and Adam moments on every rank after 5 prioritized updates" % (case, collective))


def main():
    rank, local = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
    dev = torch.device("cuda", local % torch.cuda.device_count())
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    say = (lambda s: print(s, flush=True)) if rank == 0 else (lambda s: None)
    for collective in ("nccl", "peer"):
        for case in CASES:
            check(case, collective, rank, dev, say)
    say("PER SHARDED OK")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
