"""World-size-2 tests (gloo, CPU) of the cross-rank helpers of a sharded pool (skillshot_learning_b200/learner.py):
allreduce_counters, the sum of the per-opponent counters that pool_progress reports, and ranks_agree, the one
all_gather_object after which every rank raises the same ValueError or none does.  Each test runs its two ranks under a
timeout, so a rank left waiting in a collective fails the test instead of hanging it."""
import json
import os
import socket
import time

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

WORLD = 2
CONFIG = (("n_envs", 1024), ("pool_envs", 512), ("opponents", 4), ("frames", 20), ("opponent frames", [1, 20, 20, 1]),
          ("pool_blocks", [128, 128, 128, 128]), ("collective", "peer"))


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _counters(rank):
    return torch.arange(4 * 8, dtype=torch.int64).reshape(4, 8) * (rank + 1) + 1000 * rank


def _case_sum(rank):
    from skillshot_learning_b200.learner import _broadcast_rank0, allreduce_counters
    t = _counters(rank)
    s = allreduce_counters(t, True)
    assert torch.equal(t, _counters(rank))                  # the local counters are not changed
    assert torch.equal(s, sum(_counters(r) for r in range(WORLD)))
    v = torch.full((5,), float(rank + 1))
    _broadcast_rank0(v, True)
    assert torch.equal(v, torch.ones(5))
    return "ok"


def _agree_outcome(refusal, config):
    from skillshot_learning_b200.learner import ranks_agree
    try:
        ranks_agree(refusal, config, True)
    except ValueError as e:
        msg = str(e)
    else:
        msg = None
    dist.barrier()                                          # both ranks reach the next collective
    return msg


def _case_agree(rank):
    return _agree_outcome(None, CONFIG)


def _case_differ(rank):
    cfg = dict(CONFIG)
    if rank == 1:
        cfg["pool_envs"], cfg["pool_blocks"] = 256, [64] * 4
    return _agree_outcome(None, tuple(cfg.items()))


def _case_refuse(rank):
    return _agree_outcome("pool_envs must be a multiple of 2 * 4" if rank == 1 else None, CONFIG if rank == 0 else ())


def _case_trainer(rank):
    """the trainer's constructor on a CPU device: both ranks refuse (rank 0 for the device, rank 1 already for its
    pool_envs), both raise the message of rank 0's refusal, and no rank waits"""
    import numpy as np
    from skillshot_learning_b200 import SelfPlayTrainer
    from skillshot_learning_b200.learner import A_N
    try:
        SelfPlayTrainer(64, device="cpu", opponents=[np.zeros(A_N, np.float32)] * 2, pool_envs=32 if rank == 0 else 30,
                        process_group=True)
    except ValueError as e:
        msg = str(e)
    else:
        msg = None
    dist.barrier()
    return msg


CASES = dict(sum=_case_sum, agree=_case_agree, differ=_case_differ, refuse=_case_refuse, trainer=_case_trainer)


def _worker(rank, case, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(WORLD))
    dist.init_process_group("gloo", rank=rank, world_size=WORLD)
    try:
        out = CASES[case](rank)
        with open(os.path.join(out_dir, "%s_%d.json" % (case, rank)), "w") as f:
            json.dump(out, f)
    finally:
        dist.destroy_process_group()


def _run(case, tmp_path, timeout=120.0):
    """the case on both ranks; returns their results"""
    ctx = mp.spawn(_worker, args=(case, _free_port(), str(tmp_path)), nprocs=WORLD, join=False)
    deadline = time.monotonic() + timeout
    while not ctx.join(timeout=1.0):
        if time.monotonic() > deadline:
            for p in ctx.processes:
                p.kill()
            pytest.fail("a rank did not finish within %.0f s" % timeout)
    return [json.load(open(tmp_path / ("%s_%d.json" % (case, r)))) for r in range(WORLD)]


def test_counter_sum_is_the_sum_of_the_ranks_counters(tmp_path):
    assert _run("sum", tmp_path) == ["ok", "ok"]


def test_equal_configurations_agree(tmp_path):
    assert _run("agree", tmp_path) == [None, None]


def test_a_configuration_that_differs_on_one_rank_raises_on_every_rank(tmp_path):
    m0, m1 = _run("differ", tmp_path)
    assert m0 == m1 == "rank 1 passed pool_envs = 256, rank 0 512"


def test_a_refusal_on_one_rank_raises_on_every_rank(tmp_path):
    m0, m1 = _run("refuse", tmp_path)
    assert m0 == m1 == "rank 1 refused: pool_envs must be a multiple of 2 * 4"


def test_the_sharded_pool_trainer_raises_on_every_rank_when_one_refuses(tmp_path):
    m0, m1 = _run("trainer", tmp_path)
    assert m0 == m1 == "rank 0 refused: device must be a CUDA device"
