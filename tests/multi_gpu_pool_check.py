"""Run under torchrun with 2 GPUs (tests/test_gpu_multi_pool.py launches it): a sharded pool trainer
(SelfPlayTrainer(opponents=..., process_group=True)) against single-GPU pool trainers, for a 1-frame pool (bf16 and f32)
and for a 20-frame learner against 1- and 20-frame opponents with per-env speeds and a skewed block table.  Compared with
torch.equal:

  1. each rank's rollout before any update against a single-GPU trainer with that rank's seed, weights and opponents;
  2. after rollout + update iterations with each collective, the learner's parameters, targets and Adam moments on every
     rank;
  3. pool_progress() against the figures of the all-gathered local counters, the same on every rank; reset zeroes them;
  4. rebalance_pool(): the same blocks on every rank, pfsp_blocks of the summed scores, and the restarted games against
     the single-GPU set_pool_blocks with the same table;
  5. set_pool_blocks with tables that differ by rank, and a constructor with pool_envs that differ by rank, raise on
     every rank, and nothing restarts;
  6. set_opponent with a different actor on each rank leaves rank 0's in the slot everywhere;
  7. checkpoints: fresh trainers that load each rank's file and continue reach the uninterrupted run's state."""
import os
import shutil
import sys
import tempfile

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from skillshot_learning_b200 import SelfPlayTrainer  # noqa: E402
from skillshot_learning_b200.league import _score  # noqa: E402
from skillshot_learning_b200.learner import pfsp_blocks  # noqa: E402
from tests.test_gpu_pool_frames import _actor  # noqa: E402
from tests.test_gpu_pool_speeds import _sweep  # noqa: E402

N = 1024
CASES = {
    "1-frame pool, bf16": dict(precision="bf16", opponents=[_actor(20 + k, scale=4.0) for k in range(4)], pool_envs=512),
    "1-frame pool, f32": dict(precision="f32", opponents=[_actor(20 + k, scale=4.0) for k in range(4)], pool_envs=512),
    "20-frame learner, mixed pool, speeds, skewed blocks": dict(
        precision="bf16", update_precision="bf16", frames=20, pool_envs=512, pool_blocks=[256, 128, 64, 64],
        opponents=[_actor(30, scale=4.0), _actor(31, frames=20, scale=4.0), _actor(32, scale=4.0), _actor(33, frames=20, scale=4.0)]),
}
COMMON = dict(batch_size=1024, gamma=0.95, tau=0.05, tick_limit=12, noise_group=128)


def _trainer(case, rank, dev, **kw):
    args = dict(COMMON, device=dev, seed=40 + rank, **CASES[case])
    args.update(kw)
    tr = SelfPlayTrainer(N, **args)
    if "speeds" in case:
        tr.envs.set_speeds(*_sweep(N, 31 + rank))
    return tr


def _same(a, b, stats=True):
    torch.cuda.synchronize()
    assert torch.equal(a.envs.state, b.envs.state), "env state"
    assert torch.equal(a.obs, b.obs) and torch.equal(a.actions, b.actions), "observations / actions"
    for k in ("obs", "act", "reward", "next_obs", "done"):
        assert torch.equal(getattr(a.replay, k), getattr(b.replay, k)), "ring " + k
    assert (a.replay.pos, a.replay.size) == (b.replay.pos, b.replay.size)
    if a.stack is not None:
        assert torch.equal(a.stack.stack, b.stack.stack) and torch.equal(a.rows, b.rows), "learner history"
        assert (a.stack.stack32 is None) or torch.equal(a.stack.stack32, b.stack.stack32), "learner history"
        assert (a.stack.head, a.stack.counter) == (b.stack.head, b.stack.counter)
    for x, y in zip(a.opp_stacks, b.opp_stacks):
        assert (x is None and y is None) or torch.equal(x, y), "opponent history"
    assert torch.equal(a.opponents, b.opponents), "opponents"
    if stats:
        assert torch.equal(a.pool_stats, b.pool_stats), "pool_stats"
    assert (a.envs.counter, a.networks.counter, a.pool_head, a.pool_blocks) == (b.envs.counter, b.networks.counter, b.pool_head,
                                                                                b.pool_blocks)


def _nets(tr):
    return {k: getattr(tr.networks, k) for k in ("params", "target", "adam_m", "adam_v")}


def _same_nets(a, b):
    for k, v in _nets(a).items():
        assert torch.equal(v, _nets(b)[k]), k


def _gather(obj):
    out = [None] * dist.get_world_size()
    dist.all_gather_object(out, obj)
    return out


def _raises(fn):
    try:
        fn()
    except ValueError as e:
        return str(e)
    return None


def check_case(case, collectives, rank, dev, say):
    world = dist.get_world_size()
    for c in collectives:
        tr = _trainer(case, rank, dev, process_group=True, collective=c)
        K, M = len(tr.opponents), tr.pool_envs
        # 1. before any update a rank's rollout is the single-GPU pool rollout of its envs
        solo = _trainer(case, rank, dev)
        solo.networks.set_weights(tr.networks.actor, tr.networks.critic)
        assert torch.equal(solo.opponents, tr.opponents)
        for t in (5, 9):
            tr.rollout(t)
            solo.rollout(t)
        _same(tr, solo)
        # 3. pool_progress: the figures of the summed counters, the same list on every rank
        local = _gather(tr.pool_stats.cpu())
        total = sum(local).numpy()
        want = []
        for k in range(K):
            games, wins, losses, draws, ticks = (int(v) for v in total[k, :5])
            score, se = _score(wins, draws, games)
            want.append(dict(episodes=games, wins=wins, losses=losses, draws=draws,
                             mean_ticks=ticks / games if games else float("nan"), score=score, stderr=se))
        prog = tr.pool_progress()
        assert repr(prog) == repr(want) and len(set(_gather(repr(prog)))) == 1
        assert sum(p["episodes"] for p in prog) > 0
        # 4. rebalance_pool: the same blocks everywhere, pfsp_blocks of the summed scores; the restart is the single-GPU one
        blocks = tr.rebalance_pool()
        assert blocks == pfsp_blocks([q["score"] if q["episodes"] else None for q in want], M)
        assert all(b == blocks for b in _gather(blocks))
        assert not tr.pool_stats.any(), "reset"
        solo.set_pool_blocks(blocks)
        solo.pool_stats.zero_()
        _same(tr, solo)
        tr.rollout(6)
        solo.rollout(6)
        _same(tr, solo)
        # 5. refusals: tables that differ by rank restart nothing
        state, obs = tr.envs.state.clone(), tr.obs.clone()
        other = [2] * (K - 1) + [M - 2 * (K - 1)] if rank == 1 else blocks
        msg = _raises(lambda: tr.set_pool_blocks(other))
        assert msg is not None and len(set(_gather(msg))) == 1, msg
        torch.cuda.synchronize()
        assert torch.equal(tr.envs.state, state) and torch.equal(tr.obs, obs) and tr.pool_blocks == blocks
        # 2. updates: every rank holds the same learner
        for _ in range(3):
            tr.rollout(2)
            tr.update()
        torch.cuda.synchronize()
        gathered = _gather({k: v.cpu() for k, v in _nets(tr).items()})
        for g in gathered[1:]:
            for k, v in g.items():
                assert torch.equal(v, gathered[0][k]), (c, k)
        # 7. resume: each rank's checkpoint, loaded into a fresh trainer, continues as the uninterrupted run
        path = os.path.join(tempfile.mkdtemp(prefix="pool_ckpt_"), "rank%d.pt" % rank)
        tr.save(path)
        for _ in range(2):
            tr.rollout(3)
            tr.update()
        fresh = _trainer(case, rank, dev, process_group=True, collective=c, seed=70 + rank)
        fresh.load(path)
        shutil.rmtree(os.path.dirname(path))
        for _ in range(2):
            fresh.rollout(3)
            fresh.update()
        _same(tr, fresh)
        _same_nets(tr, fresh)
        # 6. set_opponent: rank 0's actor in the slot on every rank
        k = 1
        f = tr.opp_frames[k]
        tr.set_opponent(k, _actor(100 + rank, frames=f))
        torch.cuda.synchronize()
        want_k = _actor(100, frames=f).to(dev)
        assert torch.equal(tr.opponents[k, :want_k.numel()], want_k)
        for t in (tr, fresh):
            if t.networks.peer is not None:
                t.check_exchange()
                t.networks.peer.close()
        del tr, fresh, solo
        say("%s, %s: rollout == single GPU, pool_progress / rebalance_pool / refusals / updates / resume / set_opponent ok (world %d)"
            % (case, c, world))
    # 5. a constructor with pool_envs that differ by rank raises on every rank
    msg = _raises(lambda: _trainer(case, rank, dev, process_group=True, pool_envs=512 if rank == 0 else 256))
    assert msg is not None and len(set(_gather(msg))) == 1, msg
    say("%s: constructor refusal on every rank: %s" % (case, msg))


def main(backend="nccl", collectives=("nccl", "peer")):
    rank, local = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
    dev = torch.device("cuda", local % torch.cuda.device_count())
    torch.cuda.set_device(dev)
    if backend == "nccl":
        dist.init_process_group("nccl", device_id=dev)
    else:
        dist.init_process_group(backend)
    say = (lambda s: print(s, flush=True)) if rank == 0 else (lambda s: None)
    for case in CASES:
        check_case(case, collectives, rank, dev, say)
    say("POOL SHARDED OK")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
