"""Run under torchrun with 2 GPUs (tests/test_gpu_multi_td3.py launches it): the TD3 update sharded over the ranks.

  1. the smoothing draw of rank r on its n rows (row offset r n) equals the single-GPU draw of rows [r n, (r + 1) n) of the
     global batch, for ss_td3_targets_frames and ss_td3_targets_tc (torch.equal);
  2. with each collective (NCCL all-reduce, peer exchange), sharded TD3 trainers (twin critics, delay 2, target noise)
     hold identical parameters, targets and Adam moments on every rank after rollout + update iterations (torch.equal),
     for the 12-input networks in bf16 and the 20-frame networks in float32;
  3. six sharded float32 TD3 steps on shards of a global batch follow the single-GPU steps of the whole batch up to
     summation order (2e-5)."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import learner_oracle as lo  # noqa: E402
from skillshot_learning_b200 import ActorCritic, SelfPlayTrainer  # noqa: E402
from skillshot_learning_b200 import _lib  # noqa: E402

TD3 = dict(twin_critics=True, policy_delay=2, target_noise=0.2, target_noise_clip=0.5)
CASES = {"12-input, bf16": dict(precision="bf16"), "20-frame, f32": dict(frames=20)}


def _gather(t):
    out = [torch.empty_like(t) for _ in range(dist.get_world_size())]
    dist.all_gather(out, t.contiguous())
    return out


def check_draw(rank, world, dev, say):
    g = torch.Generator(device="cpu").manual_seed(5)                  # the same global batch on every rank
    n = 3000
    N = n * world
    rng = np.random.default_rng(3)
    theta, phi, phi2 = (torch.from_numpy(x).to(dev) for x in (lo.init_actor(rng), lo.init_critic(rng), lo.init_critic(rng)))
    s2 = torch.rand((N, 12), generator=g).to(dev)
    r = (torch.rand(N, generator=g) * 2 - 1).to(dev)
    done = (torch.rand(N, generator=g) < 0.3).to(torch.uint8).to(dev)
    st = torch.cuda.current_stream(dev).cuda_stream
    L = _lib.lib
    for name in ("frames", "tc"):
        ys = []
        for rows, off in ((slice(0, N), 0), (slice(rank * n, (rank + 1) * n), rank * n)):
            m = rows.stop - rows.start
            y = torch.empty(m, device=dev)
            if name == "frames":
                rc = L.ss_td3_targets_frames(theta.data_ptr(), phi.data_ptr(), phi2.data_ptr(), 1, r[rows].data_ptr(), s2[rows].data_ptr(),
                                             done[rows].data_ptr(), 0.99, 0.2, 0.5, 17, 4, off, y.data_ptr(), m, None, 0, st)
            else:
                ws = torch.empty(_lib.td3_tc_workspace_bytes(m), dtype=torch.uint8, device=dev)
                rc = L.ss_td3_targets_tc(theta.data_ptr(), phi.data_ptr(), phi2.data_ptr(), r[rows].data_ptr(), s2[rows].data_ptr(),
                                         done[rows].data_ptr(), 0.99, 0.2, 0.5, 17, 4, off, y.data_ptr(), m, ws.data_ptr(), ws.numel(), st)
            assert rc == 0
            ys.append(y)
        # the tensor-core forwards round per 128-row tile: compare the rows of shards that start on a tile boundary
        if name == "frames" or (rank * n) % 128 == 0:
            assert torch.equal(ys[0][rank * n:(rank + 1) * n], ys[1]), name
        say("smoothing draw of rank %d's rows == the single-GPU draw of rows [%d, %d) (%s)" % (rank, rank * n, (rank + 1) * n, name))


def check_trainers(case, collective, rank, dev, say):
    kw = dict(CASES[case], device=dev, seed=40 + rank, batch_size=1024, gamma=0.95, tau=0.05, tick_limit=12, process_group=True,
              collective=collective, **TD3)
    tr = SelfPlayTrainer(512, **kw)
    for _ in range(5):
        tr.rollout(2)
        tr.update()
    torch.cuda.synchronize(dev)
    net = tr.networks
    for k in ("params", "target", "adam_m", "adam_v"):
        got = _gather(getattr(net, k))
        assert all(torch.equal(got[0], x) for x in got[1:]), (case, collective, k)
    assert net.td3_updates == 5 and net.step_actor == 2 and net.step_critic2 == 5
    if net.peer is not None:
        tr.check_exchange()
        net.peer.close()
    say("%s, %s: identical parameters, targets and Adam moments on every rank after 5 TD3 updates" % (case, collective))


def check_against_single_gpu(collective, rank, world, dev, say):
    n = 256
    rng = np.random.default_rng(9)
    theta, phi, phi2 = lo.init_actor(rng), lo.init_critic(rng), lo.init_critic(rng)
    kw = dict(device=dev, seed=7, gamma=0.99, tau=0.005, **TD3)
    sharded = ActorCritic(process_group=True, collective=collective, **kw)
    single = ActorCritic(**kw)
    for ac in (sharded, single):
        ac.set_weights(theta, phi, critic2=phi2)
    g = torch.Generator(device="cpu").manual_seed(11)
    for _ in range(6):
        s, s2 = torch.rand((n * world, 12), generator=g).to(dev), torch.rand((n * world, 12), generator=g).to(dev)
        a = (torch.rand((n * world, 2), generator=g) * 2 - 1).to(dev)
        r = (torch.rand(n * world, generator=g) * 2 - 1).to(dev)
        d = (torch.rand(n * world, generator=g) < 0.2).to(torch.uint8).to(dev)
        mine = slice(rank * n, (rank + 1) * n)
        sharded.td3_step(s[mine], a[mine], r[mine], s2[mine], d[mine])
        single.td3_step(s, a, r, s2, d)
    for v in ("actor", "critic", "critic2", "target_actor", "target_critic", "target_critic2"):
        diff = (getattr(sharded, v) - getattr(single, v)).abs().max().item()
        assert diff <= 2e-5, (v, diff)
    if sharded.peer is not None:
        sharded.peer.close()
    say("%s: six sharded TD3 steps follow the single-GPU steps of the whole batch (2e-5)" % collective)


def main():
    rank, local = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
    dev = torch.device("cuda", local % torch.cuda.device_count())
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    world = dist.get_world_size()
    say = (lambda s: print(s, flush=True)) if rank == 0 else (lambda s: None)
    check_draw(rank, world, dev, say)
    for collective in ("nccl", "peer"):
        for case in CASES:
            check_trainers(case, collective, rank, dev, say)
        check_against_single_gpu(collective, rank, world, dev, say)
    say("TD3 SHARDED OK")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
