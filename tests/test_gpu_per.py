"""Prioritized experience replay (Schaul et al. 2016, proportional; DESIGN.md section 6.16).

Without a GPU: the argument refusals of the four new entry points and of ss_ddpg_update's prioritized fields, the
constructor's and the ring loader's refusals, the header constants against _lib.py, the ranks' agreement on the four
options under gloo, and a numpy restatement of the draw against a brute-force enumeration.
On the GPU: ss_critic_grad_weighted against the unweighted entry points (==) and against a torch weighted-MSE restatement,
the prioritized draw against the numpy restatement, its distribution over 2^20 draws, the priority update and fill, the
single call against the stepwise update (==), one prioritized update on each path against the oracle, prioritized_replay
= False against the default trainer (==), and a checkpoint resume."""
import ctypes
import json
import os
import re
import socket
import time

import numpy as np
import pytest
import torch

from oracle import learner_oracle as lo
from tests import philox_ref
from tests import td3_oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
P = 1 << 20              # a 16-byte aligned stand-in for a device pointer: every call below is refused before any use
TAG_PRIORITY = 6


def _lib():
    from skillshot_learning_b200 import _lib
    return _lib


# ---------------------------------------------------------------------------------------------------------------------
# the draw, restated in numpy
# ---------------------------------------------------------------------------------------------------------------------
def per_reference(leaves, runs, batch, seed, counter, beta):
    """(ring positions drawn, weights, the eligible positions in run order, their float64 prefix P, the u of each row)"""
    pos = np.concatenate([np.arange(s, s + l) for s, l in runs]).astype(np.int64)
    lv = np.asarray(leaves, np.float32)[pos].astype(np.float64)
    pre = np.cumsum(lv)
    total = pre[-1]
    b = np.arange(batch)
    u4 = philox_ref.draw4(seed, TAG_PRIORITY, (b // 4).astype(np.uint64), np.uint64(0), counter)
    lane = b % 4
    x = np.where(lane == 0, u4[0], np.where(lane == 1, u4[1], np.where(lane == 2, u4[2], u4[3]))).astype(np.float64)
    u = (b + x * 2.0 ** -32) / batch * total
    j = np.searchsorted(pre, u, side="right")
    nz = np.nonzero(lv > 0)[0]
    j = np.minimum(j, nz[-1])
    w = ((lv[lv > 0].min() / lv[j]) ** beta).astype(np.float32)
    return pos[j], w, pos, pre, u


def _eligible_brute(capacity, size, pos, W, n, breaks):
    """the eligible ring positions by walking every filled row (tests/test_gpu_nstep.py's enumeration)"""
    oldest = (pos - size) % capacity
    cuts = {(b - oldest) % capacity for b in breaks}
    out = set()
    for o in range(size):
        last = o + (n - 1) * W
        if last < size and not any(o < c <= last for c in cuts):
            out.add((oldest + o) % capacity)
    return out


def test_numpy_draw_matches_a_brute_force_enumeration():
    from skillshot_learning_b200.learner import nstep_runs
    rng = np.random.default_rng(0)
    cases = [(96, 96, 40, 8, 1, []), (96, 60, 60, 6, 1, []), (120, 120, 48, 8, 3, [16, 88]), (200, 130, 130, 10, 4, [50]),
             (64, 64, 0, 4, 5, [8, 24, 40])]
    for capacity, size, pos, W, n, breaks in cases:
        runs = nstep_runs(capacity, size, pos, W, n, breaks)
        leaves = rng.pareto(1.5, capacity).astype(np.float32)
        leaves[rng.uniform(size=capacity) < 0.1] = 0.0
        B = 257
        src, w, order, pre, u = per_reference(leaves, runs, B, 5, 3, 0.4)
        elig = _eligible_brute(capacity, size, pos, W, n, breaks)
        assert set(order.tolist()) == elig and len(order) == len(elig)
        lv = [float(leaves[p]) for p in order]
        lmin = min(v for v in lv if v > 0)
        for b in range(B):
            acc, pick = 0.0, None
            for j, v in enumerate(lv):          # the first eligible row whose running sum exceeds u
                acc += v
                if acc > u[b]:
                    pick = j
                    break
            if pick is None:
                pick = max(j for j, v in enumerate(lv) if v > 0)
            assert src[b] == order[pick] and leaves[src[b]] > 0
            assert w[b] == np.float32((lmin / lv[pick]) ** 0.4) and 0 < w[b] <= 1
        # stratified: row b's u lies in [b, b + 1) / B of the total
        assert np.all(u >= np.arange(B) / B * pre[-1]) and np.all(u < (np.arange(B) + 1) / B * pre[-1])


# ---------------------------------------------------------------------------------------------------------------------
# refusals and constants, without a GPU
# ---------------------------------------------------------------------------------------------------------------------
def _sample_call(L, **kw):
    a = dict(ring_obs=P, ring_act=P, ring_reward=P, ring_next_obs=P, ring_done=P, capacity=1000, frames=1, tick_rows=10, n_step=1,
             gamma=0.0, runs=[(0, 500)], seed=1, counter=2, batch=16, obs=P, act=P, reward=P, next_obs=P, done=P, indices=P, steps=P,
             priority=P, scratch=P, scratch_bytes=None, beta=0.4, weights=P)
    a.update(kw)
    runs = a["runs"]
    table = None if runs is None else (ctypes.c_int64 * max(1, 2 * len(runs)))(*[v for r in runs for v in r])
    sb = int(L.ss_replay_priority_scratch_bytes(a["capacity"])) if a["scratch_bytes"] is None else a["scratch_bytes"]
    return L.ss_replay_sample_prioritized(a["ring_obs"], a["ring_act"], a["ring_reward"], a["ring_next_obs"], a["ring_done"],
                                          a["capacity"], a["frames"], a["tick_rows"], a["n_step"], a["gamma"], table,
                                          len(runs or []), a["seed"], a["counter"], a["batch"], a["obs"], a["act"], a["reward"],
                                          a["next_obs"], a["done"], a["indices"], a["steps"], a["priority"], a["scratch"], sb,
                                          a["beta"], a["weights"], None)


def test_prioritized_sampler_rejects_bad_arguments():
    L = _lib().lib
    for k in ("ring_obs", "ring_act", "ring_reward", "ring_next_obs", "ring_done", "obs", "act", "reward", "next_obs", "done", "runs",
              "priority", "scratch", "weights"):
        assert _sample_call(L, **{k: None}) == -1, k
    nan, inf = float("nan"), float("inf")
    bad = [dict(capacity=0), dict(batch=0), dict(frames=0), dict(frames=21), dict(tick_rows=0), dict(n_step=0), dict(n_step=33),
           dict(n_step=3, tick_rows=334), dict(runs=[]), dict(runs=[(0, 10)] * 17), dict(runs=[(-1, 10)]), dict(runs=[(0, 0)]),
           dict(runs=[(990, 11)]), dict(runs=[(0, 600), (100, 600)]), dict(gamma=nan), dict(beta=nan), dict(beta=inf),
           dict(beta=-0.1), dict(beta=1.5), dict(scratch_bytes=8 * 1000), dict(scratch=P + 4), dict(priority=P + 2),
           dict(weights=P + 1), dict(indices=P + 4), dict(ring_obs=P + 4), dict(next_obs=P + 8)]
    for kw in bad:
        assert _sample_call(L, **kw) == -1, kw
    assert L.ss_replay_priority_scratch_bytes(0) == -1 and L.ss_replay_priority_scratch_bytes(1000) >= 8 * 1000


def test_priority_update_fill_and_weighted_gradient_reject_bad_arguments():
    L = _lib().lib
    nan, inf = float("nan"), float("inf")

    def upd(**kw):
        a = dict(priority=P, priority_max=P, capacity=1000, indices=P, td=P, batch=16, alpha=0.6, eps=1e-6, scratch=P)
        a.update(kw)
        return L.ss_replay_priority_update(a["priority"], a["priority_max"], a["capacity"], a["indices"], a["td"], a["batch"],
                                           a["alpha"], a["eps"], a["scratch"], None)
    for kw in [dict(priority=None), dict(priority_max=None), dict(indices=None), dict(td=None), dict(scratch=None), dict(capacity=0),
               dict(batch=0), dict(alpha=-0.5), dict(alpha=nan), dict(alpha=inf), dict(eps=0.0), dict(eps=-1e-6), dict(eps=nan),
               dict(eps=inf), dict(priority=P + 2), dict(indices=P + 4), dict(td=P + 1), dict(scratch=P + 2)]:
        assert upd(**kw) == -1, kw

    def fill(**kw):
        a = dict(priority=P, priority_max=P, capacity=1000, pos=0, n=10)
        a.update(kw)
        return L.ss_replay_priority_fill(a["priority"], a["priority_max"], a["capacity"], a["pos"], a["n"], None)
    for kw in [dict(priority=None), dict(priority_max=None), dict(capacity=0), dict(pos=-1), dict(pos=1000), dict(n=0), dict(n=1001),
               dict(priority=P + 2), dict(priority_max=P + 1)]:
        assert fill(**kw) == -1, kw

    def grad(**kw):
        a = dict(phi=P, frames=1, tc=0, obs=P, act=P, y=P, w=P, td=P, keep=None, rate=0.2, n=64, n_global=0, row_offset=0, ws=P,
                 ws_bytes=1 << 24)
        a.update(kw)
        return L.ss_critic_grad_weighted(a["phi"], a["frames"], a["tc"], a["obs"], a["act"], a["y"], a["w"], a["td"], a["keep"],
                                         a["rate"], 1, 0, a["n"], a["n_global"], a["row_offset"], None, P, a["ws"], a["ws_bytes"], None)
    for tc, frames in ((0, 1), (0, 20), (1, 1), (1, 20)):
        for kw in [dict(phi=None), dict(obs=None), dict(act=None), dict(y=None), dict(ws=None), dict(n=0), dict(frames=0),
                   dict(frames=21), dict(rate=1.0), dict(rate=-0.1), dict(rate=nan), dict(w=P + 2), dict(td=P + 1), dict(phi=P + 4),
                   dict(ws_bytes=16), dict(n_global=-1), dict(row_offset=-1)]:
            args = dict(tc=tc, frames=frames)
            args.update(kw)
            assert grad(**args) == -1, (tc, frames, kw)
        if tc:
            assert grad(tc=tc, frames=frames, act=P + 4) == -1 and grad(tc=tc, frames=frames, obs=P + 8) == -1


def _update_args():
    blank = _lib().DdpgUpdateArgs()
    blank.batch, blank.size, blank.capacity, blank.step_actor, blank.step_critic = 16, 16, 16, 1, 1
    for k in ("ring_obs", "ring_act", "ring_reward", "ring_next_obs", "ring_done", "obs", "act", "reward", "next_obs", "done", "actor",
              "critic", "m_actor", "v_actor", "m_critic", "v_critic", "stats", "workspace", "indices", "priority", "priority_max",
              "priority_scratch", "priority_update_scratch", "weights", "td_abs"):
        setattr(blank, k, P)
    blank.prioritized, blank.priority_alpha, blank.priority_beta, blank.priority_eps = 1, 0.6, 0.4, 1e-6
    return blank


def test_single_call_refuses_bad_prioritized_fields():
    L = _lib().lib
    for k, v in [("sample_early", 1), ("indices", None), ("priority", None), ("priority_max", None), ("priority_scratch", None),
                 ("priority_update_scratch", None), ("weights", None), ("td_abs", None), ("priority_alpha", -1.0),
                 ("priority_alpha", float("nan")), ("priority_eps", 0.0), ("priority_eps", float("inf"))]:
        a = _update_args()
        setattr(a, k, v)
        assert L.ss_ddpg_update(ctypes.byref(a), None) == -1, k
    # a beta out of range or a short scratch is refused by the prioritized draw, the first launch, before it enqueues anything
    for k, v in [("priority_beta", 1.5), ("priority_beta", float("nan")), ("priority_scratch_bytes", 8)]:
        a = _update_args()
        a.priority_scratch_bytes = int(L.ss_replay_priority_scratch_bytes(16))
        setattr(a, k, v)
        assert L.ss_ddpg_update(ctypes.byref(a), None) == -1, k


@pytest.mark.parametrize("kw", [dict(priority_alpha=-0.1), dict(priority_alpha=float("nan")), dict(priority_beta=1.01),
                                dict(priority_beta=-0.5), dict(priority_beta=float("inf")), dict(priority_eps=0.0),
                                dict(priority_eps=-1.0), dict(priority_eps=float("nan")), dict(priority_alpha="x")])
def test_constructor_refuses_bad_priority_options_before_allocating(kw):
    from skillshot_learning_b200 import SelfPlayTrainer
    with pytest.raises(ValueError, match="priority_"):
        SelfPlayTrainer(64, device="cuda:0", prioritized_replay=True, **kw)


def test_ring_refusals_and_the_loader():
    from skillshot_learning_b200 import ReplayRing
    uni = ReplayRing(64, device="cpu")
    uni.advance(40)
    with pytest.raises(ValueError, match="prioritized=True"):
        uni.sample(8, beta=0.4)
    with pytest.raises(ValueError, match="prioritized=True"):
        uni.update_priorities([0], [1.0], 0.6, 1e-6)
    ring = ReplayRing(64, device="cpu", prioritized=True)
    ring.size = 40
    for beta in (-0.1, 1.5, float("nan"), "x"):
        with pytest.raises(ValueError, match="beta"):
            ring.sample(8, beta=beta)
    with pytest.raises(ValueError, match="indices must be None"):
        ring.sample(8, beta=0.4, indices=[1] * 8)
    with pytest.raises(ValueError, match="priority_eps"):
        ring.update_priorities([0], [1.0], 0.6, 0.0)
    # a checkpoint of a uniform ring loads with every leaf and priority_max at 1.0; a uniform ring ignores the leaves
    sd = uni.state_dict()
    assert "priority" not in sd
    ring.priority.fill_(3.0)
    ring.load_state_dict(sd)
    assert bool((ring.priority == 1.0).all()) and float(ring.priority_max) == 1.0 and ring.size == 40
    ring.priority[5] = 7.0
    ring.priority_max.fill_(7.0)
    sd = ring.state_dict()
    assert torch.equal(sd["priority"], ring.priority) and float(sd["priority_max"]) == 7.0
    other = ReplayRing(64, device="cpu", prioritized=True)
    other.load_state_dict(sd)
    assert torch.equal(other.priority, ring.priority) and float(other.priority_max) == 7.0
    uni2 = ReplayRing(64, device="cpu")
    uni2.load_state_dict(sd)
    assert not hasattr(uni2, "priority")
    sd["priority"] = torch.ones(32)
    with pytest.raises(ValueError, match="priority leaves"):
        other.load_state_dict(sd)


def test_header_constants_match_the_python_mirror():
    _l = _lib()
    text = open(os.path.join(ROOT, "include", "skillshot_b200.h")).read()
    assert int(re.search(r"#define\s+SS_TAG_PRIORITY\s+(\d+)", text).group(1)) == _l.TAG_PRIORITY == TAG_PRIORITY
    rng_h = open(os.path.join(ROOT, "skillshot_learning_b200", "csrc", "ss_rng.cuh")).read()
    assert int(re.search(r"kTagPriority\s*=\s*(\d+)", rng_h).group(1)) == TAG_PRIORITY
    tags = [int(v) for v in re.findall(r"constexpr uint32_t kTag\w+\s*=\s*(\d+)", rng_h)]
    assert len(tags) == len(set(tags))                  # a tag of its own
    names = [f[0] for f in _l.DdpgUpdateArgs._fields_]
    assert names[-11:] == ["prioritized", "priority", "priority_max", "priority_scratch", "priority_scratch_bytes",
                           "priority_update_scratch", "priority_alpha", "priority_beta", "priority_eps", "weights", "td_abs"]


# ---- the agreement of the ranks on the four options (gloo, world size 2, under a timeout) ----------------------------
WORLD = 2


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _gloo_case(rank, case):
    import torch.distributed as dist
    from skillshot_learning_b200 import SelfPlayTrainer
    try:
        if case == "differ":           # rank 1 passes another beta; both are valid
            SelfPlayTrainer(64, device="cpu", process_group=True, prioritized_replay=True, priority_beta=0.4 + 0.2 * rank)
        elif case == "flag":           # rank 1 trains uniformly
            SelfPlayTrainer(64, device="cpu", process_group=True, prioritized_replay=rank == 0)
        elif case == "refuse":         # rank 1 refuses its eps
            SelfPlayTrainer(64, device="cpu", process_group=True, prioritized_replay=True, priority_eps=0.0 if rank else 1e-6)
        else:                          # both agree: the constructor goes on and fails later, on the CPU device
            SelfPlayTrainer(64, device="cpu", process_group=True, prioritized_replay=True)
    except (ValueError, RuntimeError, AssertionError) as e:
        msg = "%s: %s" % (type(e).__name__, str(e).splitlines()[0])
    else:
        msg = None
    dist.barrier()
    return msg


def _worker(rank, case, port, out_dir):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(WORLD))
    dist.init_process_group("gloo", rank=rank, world_size=WORLD)
    try:
        out = _gloo_case(rank, case)
        with open(os.path.join(out_dir, "%s_%d.json" % (case, rank)), "w") as f:
            json.dump(out, f)
    finally:
        dist.destroy_process_group()


def _run(case, tmp_path, timeout=120.0):
    import torch.multiprocessing as mp
    ctx = mp.spawn(_worker, args=(case, _free_port(), str(tmp_path)), nprocs=WORLD, join=False)
    deadline = time.monotonic() + timeout
    while not ctx.join(timeout=1.0):
        if time.monotonic() > deadline:
            for p in ctx.processes:
                p.kill()
            pytest.fail("a rank did not finish within %.0f s" % timeout)
    return [json.load(open(tmp_path / ("%s_%d.json" % (case, r)))) for r in range(WORLD)]


def test_ranks_agree_on_the_priority_options(tmp_path):
    m0, m1 = _run("differ", tmp_path)
    assert m0 == m1 == "ValueError: rank 1 passed priority_beta = 0.6000000000000001, rank 0 0.4"
    m0, m1 = _run("flag", tmp_path)
    assert m0 == m1 == "ValueError: rank 1 passed prioritized_replay = False, rank 0 True"
    m0, m1 = _run("refuse", tmp_path)
    assert m0 == m1 == "ValueError: rank 1 refused: priority_eps must be finite and > 0, got 0.0"
    m0, m1 = _run("agree", tmp_path)
    assert m0 == m1 and "priority" not in (m0 or "")


# ---------------------------------------------------------------------------------------------------------------------
# on the GPU
# ---------------------------------------------------------------------------------------------------------------------
gpu = pytest.mark.gpu
DEV = "cuda:0"


def _rand_batch(rng, n, frames):
    s = rng.uniform(0, 1, (n, 12 * frames)).astype(np.float32)
    a = rng.uniform(-1, 1, (n, 2)).astype(np.float32)
    y = rng.uniform(-1, 1, n).astype(np.float32)
    return s, a, y


def _net(frames, tc, seed=3):
    from skillshot_learning_b200 import ActorCritic
    ac = ActorCritic(device=DEV, seed=seed, frames=frames, update_precision="bf16" if tc else "f32")
    rng = np.random.default_rng(seed)
    ac.set_weights(lo.init_actor(rng, frames), lo.init_critic(rng, frames))
    return ac


FAMILIES = [(1, False), (20, False), (1, True), (20, True)]


@gpu
@pytest.mark.parametrize("frames,tc", FAMILIES)
def test_weighted_gradient_with_unit_or_no_weights_is_the_unweighted_one(frames, tc):
    rng = np.random.default_rng(frames)
    n = 3000
    s, a, y = _rand_batch(rng, n, frames)
    res = []
    for kw in ({}, dict(weights=None, td_abs_out=None), dict(weights=torch.ones(n, device=DEV)),
               dict(td_abs_out=torch.empty(n, device=DEV)), dict(weights=torch.ones(n, device=DEV), td_abs_out=torch.empty(n, device=DEV))):
        ac = _net(frames, tc)
        g = ac.critic_grad(s, a, y, **kw).clone()
        res.append((g, ac.stats[0].clone()))
    for g, sse in res[1:]:
        assert torch.equal(g, res[0][0]) and torch.equal(sse, res[0][1])


def weighted_critic_grad(phi, s, a, y, w, keep, rate=0.2):
    """the learner oracle's critic gradient of the row-weighted loss mean(w (q - y)^2), and |q - y|"""
    p = torch.tensor(np.asarray(phi, np.float32)).requires_grad_(True)
    q = lo.critic_forward_t(p, torch.tensor(s), torch.tensor(a), None if keep is None else torch.tensor(keep, dtype=torch.float32), rate)
    e = q - torch.tensor(y)
    ((e ** 2 * torch.tensor(w)).sum() / len(y)).backward()
    return p.grad.numpy().copy(), np.abs(e.detach().numpy())


@gpu
@pytest.mark.parametrize("frames,tc", FAMILIES)
def test_weighted_gradient_tracks_a_torch_restatement(frames, tc):
    rng = np.random.default_rng(10 + frames)
    n = 2000
    s, a, y = _rand_batch(rng, n, frames)
    w = rng.uniform(0.05, 1.0, n).astype(np.float32)
    keep = (rng.uniform(size=(n, 256)) >= 0.2).astype(np.uint8)
    ac = _net(frames, tc)
    phi = ac.critic.cpu().numpy()
    td = torch.empty(n, device=DEV)
    g = ac.critic_grad(s, a, y, keep=keep, weights=torch.from_numpy(w), td_abs_out=td).cpu().numpy()
    want, e = weighted_critic_grad(phi, s, a, y, w, keep)
    tol = 2e-2 if tc else 2e-5
    assert np.abs(g - want).max() <= tol * np.abs(want).max()
    np.testing.assert_allclose(td.cpu().numpy(), e, rtol=0, atol=(2e-2 if tc else 2e-5) * max(1.0, np.abs(e).max()))
    unweighted = _net(frames, tc).critic_grad(s, a, y, keep=keep).cpu().numpy()
    assert np.abs(unweighted - want).max() > 10 * tol * np.abs(want).max()      # the weights matter


def _trainer(**kw):
    from skillshot_learning_b200 import SelfPlayTrainer
    base = dict(device=DEV, seed=3, batch_size=512, gamma=0.99, tau=0.005, reward_mode="terminal", tick_limit=40)
    base.update(kw)
    return SelfPlayTrainer(base.pop("n_envs", 256), **base)


def _skew_leaves(ring, seed):
    rng = np.random.default_rng(seed)
    lv = rng.pareto(1.2, ring.capacity).astype(np.float32) + np.float32(1e-3)
    lv[rng.uniform(size=ring.capacity) < 0.05] = 0.0
    ring.priority.copy_(torch.from_numpy(lv))
    return lv


def _check_draw(ring, batch, beta, n=1, gamma=0.0):
    from skillshot_learning_b200.learner import nstep_runs
    runs = [(0, ring.size)] if n == 1 else nstep_runs(ring.capacity, ring.size, ring.pos, ring.tick_rows, n, ring.breaks)
    lv = ring.priority.cpu().numpy()
    counter = ring.counter
    b = ring.sample(batch, n_step=n, gamma=gamma, beta=beta)
    ring.counter = counter
    again = ring.sample(batch, n_step=n, gamma=gamma, beta=beta)
    for k in b:
        assert torch.equal(b[k], again[k]), k
    src, w, order, pre, u = per_reference(lv, runs, batch, ring.seed, counter, beta)
    idx = b["indices"].cpu().numpy()
    where = {p: j for j, p in enumerate(order.tolist())}
    j = np.array([where[int(i)] for i in idx])
    tol = 1e-12 * pre[-1]
    lo_edge = np.where(j > 0, pre[np.maximum(j - 1, 0)], 0.0)
    assert np.all(u >= lo_edge - tol) and np.all((u < pre[j] + tol) | (j == np.nonzero(lv[order] > 0)[0][-1]))
    assert np.all(lv[idx] > 0)
    lmin = lv[order][lv[order] > 0].min()
    np.testing.assert_allclose(b["weights"].cpu().numpy(), (np.float64(lmin) / lv[idx].astype(np.float64)) ** beta, rtol=1e-6)
    obs, act = ring.obs.cpu().numpy(), ring.act.cpu().numpy()
    assert np.array_equal(b["obs"].cpu().numpy(), obs[idx]) and np.array_equal(b["act"].cpu().numpy(), act[idx])
    if n == 1:
        assert np.array_equal(b["reward"].cpu().numpy(), ring.reward.cpu().numpy()[idx])
        assert np.array_equal(b["next_obs"].cpu().numpy(), ring.next_obs.cpu().numpy()[idx])
        assert np.array_equal(b["done"].cpu().numpy(), ring.done.cpu().numpy()[idx])
    else:
        d, r = ring.done.cpu().numpy(), ring.reward.cpu().numpy()
        got_r, got_k, got_d = b["reward"].cpu().numpy(), b["steps"].cpu().numpy(), b["done"].cpu().numpy()
        got_s2, s2 = b["next_obs"].cpu().numpy(), ring.next_obs.cpu().numpy()
        gm = np.float32(gamma)
        for i, s0 in enumerate(idx):
            row, sm, g, k = int(s0), r[int(s0)], np.float32(1), 1
            while k < n and not d[row]:
                row = (row + ring.tick_rows) % ring.capacity
                g = np.float32(g * gm)
                sm = np.float32(sm + np.float32(g * r[row]))
                k += 1
            assert got_r[i] == sm and got_k[i] == k and got_d[i] == d[row] and np.array_equal(got_s2[i], s2[row])
    return b


@gpu
@pytest.mark.parametrize("n", [1, 3, 5])
def test_prioritized_draw_matches_the_numpy_restatement(n):
    # self-play, wrapped ring, a store=False break (n-step); then a partly filled frame-stacked ring
    t = _trainer(n_step=n, n_envs=1024, replay_capacity=2048 * 30, prioritized_replay=True)
    t.rollout(25)
    t.rollout(2, store=False)
    t.rollout(20)
    assert t.replay.size == t.replay.capacity and t.replay.pos != 0 and int(t.replay.done.sum()) > 0
    _skew_leaves(t.replay, n)
    _check_draw(t.replay, 65536, 0.4, n, 0.99)
    t = _trainer(n_step=n, frames=20, n_envs=128, replay_capacity=256 * 40, prioritized_replay=True)
    t.rollout(13)
    assert t.replay.size < t.replay.capacity
    _skew_leaves(t.replay, n + 7)
    _check_draw(t.replay, 4099, 1.0, n, 0.9)


@gpu
def test_two_to_the_twenty_draws_follow_the_leaves():
    from scipy.stats import chisquare
    from skillshot_learning_b200 import ReplayRing
    from skillshot_learning_b200.learner import nstep_runs
    W, n = 16, 3
    ring = ReplayRing(W * 300, device=DEV, seed=9, tick_rows=W, prioritized=True)
    rng = np.random.default_rng(9)
    for t in range(340):
        ring.push(*(torch.from_numpy(rng.uniform(-1, 1, (W, k)).astype(np.float32)) for k in (12, 2)), torch.zeros(W),
                  torch.zeros((W, 12)))
        if t % 47 == 0:
            ring.mark_break()
    lv = rng.choice([0.0, 0.01, 1.0, 30.0], ring.capacity, p=[0.05, 0.35, 0.5, 0.1]).astype(np.float32)
    ring.priority.copy_(torch.from_numpy(lv))
    runs = nstep_runs(ring.capacity, ring.size, ring.pos, W, n, ring.breaks)
    eligible = np.zeros(ring.capacity, bool)
    for s, l in runs:
        eligible[s:s + l] = True
    assert 1 < len(runs) and eligible.sum() < ring.size
    counts = np.zeros(ring.capacity, np.int64)
    for _ in range(4):
        b = ring.sample(1 << 18, n_step=n, gamma=0.9, beta=0.5)
        counts += np.bincount(b["indices"].cpu().numpy(), minlength=ring.capacity)
    assert counts.sum() == 1 << 20 and counts[~eligible].sum() == 0 and counts[lv == 0].sum() == 0
    live = eligible & (lv > 0)
    expect = lv[live].astype(np.float64) / lv[live].astype(np.float64).sum() * (1 << 20)
    assert chisquare(counts[live], expect).pvalue > 1e-3


@gpu
def test_priority_update_takes_the_last_duplicate_and_raises_the_maximum():
    from skillshot_learning_b200 import ReplayRing
    ring = ReplayRing(1000, device=DEV, prioritized=True)
    ring.advance(1000)
    assert bool((ring.priority == 1.0).all())
    rng = np.random.default_rng(3)
    B = 20000
    idx = rng.integers(0, 1000, B)                    # about 20 occurrences of every position
    td = rng.uniform(0, 3, B).astype(np.float32)
    ring.update_priorities(torch.from_numpy(idx), torch.from_numpy(td), 0.6, 1e-6)
    want = np.ones(1000, np.float32)
    leaf = np.power(np.abs(td) + np.float32(1e-6), np.float32(0.6), dtype=np.float32)
    for b in range(B):
        want[idx[b]] = leaf[b]                        # the largest batch position wins
    np.testing.assert_allclose(ring.priority.cpu().numpy(), want, rtol=2e-7, atol=0)
    assert float(ring.priority_max) == float(ring.priority.max()) > 1.0
    # a smaller update leaves priority_max where it was; a fill writes it
    top = float(ring.priority_max)
    ring.update_priorities(torch.tensor([5]), torch.tensor([0.0]), 0.6, 1e-6)
    assert float(ring.priority_max) == top and float(ring.priority[5]) < 1e-3
    ring.advance(3)
    assert bool((ring.priority[:3] == top).all())


@gpu
@pytest.mark.parametrize("kind", ["self-play", "frames", "pool"])
def test_rollouts_fill_exactly_the_new_rows(kind):
    kw = dict(prioritized_replay=True)
    if kind == "frames":
        kw.update(frames=20, n_envs=128)
    if kind == "pool":
        rng = np.random.default_rng(1)
        kw.update(opponents=[lo.init_actor(rng), lo.init_actor(rng, 20)], pool_envs=128)
    t = _trainer(**kw)
    ring = t.replay
    rows = t.learner_rows
    t.rollout(3)
    assert bool((ring.priority[:3 * rows] == 1.0).all()) and bool((ring.priority[3 * rows:] == 0.0).all())
    ring.priority_max.fill_(2.5)
    t.rollout(7)                                      # 10 ticks of 8 fit: wraps over the first two
    lv = ring.priority.cpu().numpy()
    assert ring.pos == 2 * rows and np.all(lv[:2 * rows] == 2.5) and np.all(lv[2 * rows:3 * rows] == 1.0)
    assert np.all(lv[3 * rows:] == 2.5)
    t.rollout_tick()
    assert np.all(ring.priority.cpu().numpy()[2 * rows:3 * rows] == 2.5)


def _same_state(a, b):
    na, nb = a.networks, b.networks
    for k in ("params", "target", "adam_m", "adam_v"):
        assert torch.equal(getattr(na, k), getattr(nb, k)), k
    assert (na.step_actor, na.step_critic, na.counter) == (nb.step_actor, nb.step_critic, nb.counter)
    for k in ("obs", "act", "reward", "next_obs", "done"):
        assert torch.equal(getattr(a.replay, k), getattr(b.replay, k)), k
    assert (a.replay.pos, a.replay.size, a.replay.counter) == (b.replay.pos, b.replay.size, b.replay.counter)
    if a.replay.prioritized:
        assert torch.equal(a.replay.priority, b.replay.priority) and torch.equal(a.replay.priority_max, b.replay.priority_max)


@gpu
@pytest.mark.parametrize("precision", ["f32", "bf16"])
def test_single_call_equals_the_stepwise_update(precision, monkeypatch):
    lib = _lib().lib
    calls = []
    real = lib.ss_ddpg_update
    monkeypatch.setattr(lib, "ss_ddpg_update", lambda *x: calls.append(1) or real(*x))
    a, b = (_trainer(prioritized_replay=True, precision=precision) for _ in range(2))
    for _ in range(10):
        for t in (a, b):
            t.rollout(2)
        a.update()
        b.update_stepwise()
    _same_state(a, b)
    assert len(calls) == 10 and float(a.replay.priority_max) > 1.0


@gpu
@pytest.mark.parametrize("path", ["single", "stepwise", "frames", "pool", "td3"])
def test_uniform_option_is_the_default_trainer_bit_for_bit(path, monkeypatch):
    lib = _lib().lib
    calls = []
    real = lib.ss_ddpg_update
    monkeypatch.setattr(lib, "ss_ddpg_update", lambda *x: calls.append(1) or real(*x))
    kw = dict(precision="bf16")
    if path == "frames":
        kw.update(frames=20, n_envs=128)
    if path == "pool":
        rng = np.random.default_rng(1)
        kw.update(opponents=[lo.init_actor(rng), lo.init_actor(rng, 20)], pool_envs=128)
    if path == "td3":
        kw.update(twin_critics=True, policy_delay=2, target_noise=0.2)
    a, b = _trainer(**kw), _trainer(prioritized_replay=False, **kw)
    assert not b.replay.prioritized and not hasattr(b.replay, "priority")
    for _ in range(20):
        for t in (a, b):
            t.rollout(2)
            t.update_stepwise() if path == "stepwise" else t.update()
    _same_state(a, b)
    assert len(calls) == (40 if path in ("single", "pool") else 0)
    assert set(b.state_dict()["replay"]) == set(a.state_dict()["replay"])


class PerOracle(td3_oracle.TD3Oracle):
    """TD3Oracle with prioritized replay's weighted critic loss; update() also returns critic 1's |q - y|"""

    def update(self, s, a, r, s2, done, eps, keep1, keep2=None, w=None):
        y = td3_oracle.td3_targets(self.theta_t, self.phi_t, self.phi2_t, r, s2, done, self.gamma, eps, self.sigma, self.clip)
        delayed = (self.updates + 1) % self.policy_delay == 0
        tau = self.tau if delayed else 0.0
        g, td = weighted_critic_grad(self.phi, s, a, y, w, keep1, self.dropout)
        self.phi = self.opt_critic.step(self.phi, g)
        self.phi_t = lo.soft_update(self.phi_t, self.phi, tau)
        if self.phi2 is not None:
            g, _ = weighted_critic_grad(self.phi2, s, a, y, w, keep2, self.dropout)
            self.phi2 = self.opt_critic2.step(self.phi2, g)
            self.phi2_t = lo.soft_update(self.phi2_t, self.phi2, tau)
        if delayed:
            g, _ = lo.actor_grad(self.theta, self.phi, s)
            self.theta = self.opt_actor.step(self.theta, g)
            self.theta_t = lo.soft_update(self.theta_t, self.theta, tau)
        self.updates += 1
        return y, td


@gpu
@pytest.mark.parametrize("path", ["single", "stepwise", "frames", "pool", "td3", "nstep"])
def test_one_prioritized_update_tracks_the_oracle(path):
    from skillshot_learning_b200.learner import nstep_discount
    kw = dict(prioritized_replay=True, priority_alpha=0.7, priority_beta=0.5, priority_eps=1e-3, batch_size=384)
    if path == "frames":
        kw.update(frames=20, n_envs=128)
    if path == "pool":
        rng = np.random.default_rng(1)
        kw.update(opponents=[lo.init_actor(rng), lo.init_actor(rng)], pool_envs=128)
    if path == "td3":
        kw.update(twin_critics=True, policy_delay=1)
    if path == "nstep":
        kw.update(n_step=3)
    t = _trainer(**kw)
    t.rollout(6)
    _skew_leaves(t.replay, 4)
    net = t.networks
    frames = t.frames
    twin = path == "td3"
    orc = PerOracle(net.actor.cpu().numpy(), net.critic.cpu().numpy(), net.critic2.cpu().numpy() if twin else None,
                    gamma=nstep_discount(0.99, 3) if path == "nstep" else 0.99, tau=0.005, policy_delay=1, sigma=0.0, dropout=0.2)
    orc.theta_t, orc.phi_t = net.target_actor.cpu().numpy(), net.target_critic.cpu().numpy()
    if twin:
        orc.phi2_t = net.target_critic2.cpu().numpy()
    k = net.counter
    if path == "stepwise":
        t.update_stepwise()
    else:
        t.update()
    b = t._batch
    B = t.batch_size
    keeps = [philox_ref.dropout_keep(B, net.seed, k + j, 0.2).astype(np.float32) for j in (0, 1)]
    s, a, r, s2, d, w = (b[x].cpu().numpy() for x in ("obs", "act", "reward", "next_obs", "done", "weights"))
    assert s.shape[1] == 12 * frames and w.min() > 0 and w.max() <= 1 and w.min() < 1
    y, td = orc.update(s, a, r, s2, d, None, keeps[0], keeps[1] if twin else None, w=w)
    pairs = [(net.actor, orc.theta), (net.critic, orc.phi), (net.target_actor, orc.theta_t), (net.target_critic, orc.phi_t)]
    if twin:
        pairs += [(net.critic2, orc.phi2)]
    for got, want in pairs:
        np.testing.assert_allclose(got.cpu().numpy(), want, rtol=0, atol=2e-5)
    np.testing.assert_allclose(b["td_abs"].cpu().numpy(), td, rtol=0, atol=2e-5 * max(1.0, np.abs(td).max()))
    idx = b["indices"].cpu().numpy()
    last = {}
    for i, p in enumerate(idx):
        last[int(p)] = i
    pos = np.array(sorted(last))
    winner = np.array([last[p] for p in pos])
    leaves = t.replay.priority.cpu().numpy()[pos]
    # (|delta| + eps)^alpha of the oracle's delta (at the tolerance its |delta| carries), and of the kernel's own |delta|
    np.testing.assert_allclose(leaves, np.power(td[winner].astype(np.float64) + 1e-3, 0.7), rtol=2e-2)
    np.testing.assert_allclose(leaves, np.power(b["td_abs"].cpu().numpy()[winner].astype(np.float64) + 1e-3, 0.7), rtol=1e-6)


@gpu
def test_checkpoint_resumes_bit_identically_and_old_checkpoints_load(tmp_path):
    kw = dict(prioritized_replay=True, precision="bf16")
    a = _trainer(**kw)
    for _ in range(3):
        a.rollout(2)
        a.update()
    a.save(str(tmp_path / "ck.pt"))
    b = _trainer(**kw)
    b.load(str(tmp_path / "ck.pt"))
    assert torch.equal(a.replay.priority, b.replay.priority)
    for i in range(6):
        for t in (a, b):
            t.priority_beta = 0.4 + 0.1 * i           # annealed by the caller
            t.rollout(2)
            t.update()
    _same_state(a, b)
    c = _trainer(precision="bf16")
    c.rollout(4)
    c.save(str(tmp_path / "old.pt"))
    d = _trainer(**kw)
    d.load(str(tmp_path / "old.pt"))
    assert d.replay.size == c.replay.size and bool((d.replay.priority == 1.0).all()) and float(d.replay.priority_max) == 1.0
    d.update()
