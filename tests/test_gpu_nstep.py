"""n-step returns drawn from the replay ring (no reference code, DESIGN.md section 6.15).

Without a GPU: nstep_runs against a brute-force enumeration of the eligible rows, the ring's own bookkeeping of its breaks
against a restatement in absolute write counts, the argument refusals of ss_replay_sample_nstep / ss_ddpg_update and of the
constructors, the header constants against _lib.py, and the ranks' agreement on n_step under gloo.
On the GPU, compared with ==: n = 1 against ss_replay_sample_frames, n_step = 1 trainers against default trainers, n = 3 and 5
against a numpy restatement of the walk on rings filled by real rollouts, and a checkpoint resume; over 10^6 draws, the
support and uniformity of the draw; n-step updates against the learner oracle (tests/td3_oracle.py) at section 6.2's
tolerances."""
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


def _lib():
    from skillshot_learning_b200 import _lib
    return _lib


# ---------------------------------------------------------------------------------------------------------------------
# without a GPU
# ---------------------------------------------------------------------------------------------------------------------
def _eligible_brute(capacity, size, pos, W, n, breaks):
    """the eligible ring positions, by walking every filled row: the walk of the row of write order o (0 = oldest) visits
    o, o + W, ..., o + (n - 1) W and must stay below `size` and not step over a break"""
    oldest = (pos - size) % capacity
    cuts = {(b - oldest) % capacity for b in breaks}
    out = set()
    for o in range(size):
        last = o + (n - 1) * W
        if last < size and not any(o < c <= last for c in cuts):
            out.add((oldest + o) % capacity)
    return out


def _intervals(rows, capacity, size, pos):
    """maximal runs of ring positions of `rows`, each with the write order of its first row"""
    oldest = (pos - size) % capacity
    runs, start = [], None
    for p in range(capacity + 1):
        inside = p < capacity and p in rows
        if inside and start is None:
            start = p
        if not inside and start is not None:
            runs.append((start, p - start, (start - oldest) % capacity))
            start = None
    return runs


def _expected_runs(capacity, size, pos, W, n, breaks):
    runs = _intervals(_eligible_brute(capacity, size, pos, W, n, breaks), capacity, size, pos)
    if n == 1 and runs:
        assert runs == [(0, size, runs[0][2])]
    m = _lib().REPLAY_MAX_RUNS
    if len(runs) > m:
        runs = sorted(sorted(runs, key=lambda r: r[2])[-m:])
    return [(s, l) for s, l, _ in runs]


def test_nstep_runs_against_brute_force():
    from skillshot_learning_b200.learner import nstep_runs
    rng = np.random.default_rng(0)
    seen_wrap = seen_partial = seen_many = 0
    for case in range(3000):
        W = int(rng.integers(1, 9))
        capacity = W * int(rng.integers(1, 40)) + (int(rng.integers(0, W)) if case % 3 == 0 else 0)
        n = int(rng.integers(1, 6))
        full = rng.uniform() < 0.5
        size = capacity if full else int(rng.integers(0, capacity + 1))
        pos = int(rng.integers(0, capacity)) if full else size % capacity
        nb = int(rng.integers(0, 5))
        if case % 10 == 0:               # more breaks than runs
            W, n = int(rng.integers(1, 4)), int(rng.integers(2, 4))
            capacity = size = W * int(rng.integers(60, 120))
            pos, nb = int(rng.integers(0, capacity)), int(rng.integers(20, 60))
        breaks = [int(b) for b in rng.integers(0, capacity, size=nb)]
        got = nstep_runs(capacity, size, pos, W, n, breaks)
        want = _expected_runs(capacity, size, pos, W, n, breaks)
        assert got == want, (capacity, size, pos, W, n, breaks)
        seen_wrap += full and pos != 0
        seen_partial += not full and 0 < size < capacity
        seen_many += len(_intervals(_eligible_brute(capacity, size, pos, W, n, breaks), capacity, size, pos)) > len(got)
    assert seen_wrap > 100 and seen_partial > 100 and seen_many > 10
    # n = 1: one run (0, size) whatever the breaks
    assert nstep_runs(100, 100, 37, 10, 1, [10, 50, 90]) == [(0, 100)]
    assert nstep_runs(100, 60, 60, 10, 1, [10, 50]) == [(0, 60)]
    # fewer than n ticks stored: nothing to draw
    assert nstep_runs(100, 20, 20, 10, 3, []) == [] and nstep_runs(100, 30, 30, 10, 3, []) == [(0, 10)]


def test_ring_keeps_its_breaks_as_absolute_write_counts_would():
    """A ring on the host (no device writes): blocks of W rows written tick by tick with breaks in between; its
    eligible_runs equal the runs of the rows eligible by absolute write counts, where a break at count T_b excludes the
    rows a with a < T_b <= a + (n - 1) W and the rows still stored are [T - size, T)."""
    from skillshot_learning_b200 import ReplayRing
    rng = np.random.default_rng(1)
    for case in range(200):
        W = int(rng.integers(1, 6))
        cap = W * int(rng.integers(2, 12)) + (int(rng.integers(0, W)) if case % 2 else 0)
        ring = ReplayRing(cap, device="cpu", tick_rows=W)
        T, marks = 0, []
        for _ in range(int(rng.integers(1, 60))):
            if rng.uniform() < 0.25:
                ring.mark_break()
                if T > 0:
                    marks.append(T)
            else:
                ring.advance(W)
                T += W
            size = min(T, cap)
            assert (ring.pos, ring.size) == (T % cap, size)
            for n in (1, 2, 3):
                if n * W > cap:
                    continue
                rows = {a % cap for a in range(T - size, T)
                        if a + (n - 1) * W < T and not any(a < tb <= a + (n - 1) * W for tb in marks)}
                runs = _intervals(rows, cap, size, T % cap)
                m = _lib().REPLAY_MAX_RUNS
                if len(runs) > m:
                    runs = sorted(sorted(runs, key=lambda r: r[2])[-m:])
                assert ring.eligible_runs(n) == [(s, l) for s, l, _ in runs], (case, n)
            assert len(ring.breaks) <= cap


def _nstep_call(L, **kw):
    a = dict(ring_obs=P, ring_act=P, ring_reward=P, ring_next_obs=P, ring_done=P, capacity=1000, frames=1, tick_rows=10, n_step=3,
             gamma=0.99, runs=[(0, 500)], n_runs=None, seed=1, counter=2, batch=16, obs=P, act=P, reward=P, next_obs=P, done=P,
             indices=P, steps=P)
    a.update(kw)
    import ctypes
    runs = a["runs"]
    table = None if runs is None else (ctypes.c_int64 * max(1, 2 * len(runs)))(*[v for r in runs for v in r])
    n_runs = len(runs or []) if a["n_runs"] is None else a["n_runs"]
    return L.ss_replay_sample_nstep(a["ring_obs"], a["ring_act"], a["ring_reward"], a["ring_next_obs"], a["ring_done"], a["capacity"],
                                    a["frames"], a["tick_rows"], a["n_step"], a["gamma"], table, n_runs, a["seed"], a["counter"],
                                    a["batch"], a["obs"], a["act"], a["reward"], a["next_obs"], a["done"], a["indices"], a["steps"],
                                    None)


def test_nstep_sampler_rejects_bad_arguments():
    L = _lib().lib
    for k in ("ring_obs", "ring_act", "ring_reward", "ring_next_obs", "ring_done", "obs", "act", "reward", "next_obs", "done", "runs"):
        assert _nstep_call(L, **{k: None}) == -1, k
    bad = [dict(capacity=0), dict(batch=0), dict(frames=0), dict(frames=21), dict(tick_rows=0), dict(n_step=0), dict(n_step=33),
           dict(n_step=3, tick_rows=334), dict(runs=[]), dict(runs=[(0, 10)] * 17), dict(runs=[(-1, 10)]), dict(runs=[(0, 0)]),
           dict(runs=[(990, 11)]), dict(runs=[(1000, 1)]), dict(runs=[(0, 10), (20, -3)]), dict(gamma=float("nan")),
           dict(gamma=float("inf")), dict(ring_obs=P + 4), dict(next_obs=P + 8), dict(capacity=1 << 33, runs=[(0, 1 << 32)]),
           dict(runs=[(0, 10)], n_runs=2)]
    for kw in bad:
        assert _nstep_call(L, **kw) == -1, kw
    # ss_ddpg_update refuses an n_step out of range before anything else
    import ctypes
    blank = _lib().DdpgUpdateArgs()
    blank.batch, blank.size, blank.capacity, blank.step_actor, blank.step_critic = 16, 16, 16, 1, 1
    for k in ("ring_obs", "ring_act", "ring_reward", "ring_next_obs", "ring_done", "obs", "act", "reward", "next_obs", "done", "actor",
              "critic", "m_actor", "v_actor", "m_critic", "v_critic", "stats", "workspace"):
        setattr(blank, k, P)
    for n in (-1, 33):
        blank.n_step = n
        assert L.ss_ddpg_update(ctypes.byref(blank), None) == -1


@pytest.mark.parametrize("n_step", [0, 33, -2, 1.5, True, "3", None])
def test_constructors_reject_a_bad_n_step_before_allocating(n_step):
    from skillshot_learning_b200 import SelfPlayTrainer
    with pytest.raises(ValueError, match="n_step must be an integer"):
        SelfPlayTrainer(64, device="cuda:0", n_step=n_step)


def test_capacity_below_n_ticks_and_rings_without_tick_rows_are_refused():
    from skillshot_learning_b200 import ReplayRing, SelfPlayTrainer
    from skillshot_learning_b200.learner import A_N
    with pytest.raises(ValueError, match="replay capacity of at least 384"):
        SelfPlayTrainer(64, device="cuda:0", replay_capacity=256, n_step=3)
    with pytest.raises(ValueError, match="replay capacity of at least 320"):     # a pool: 64 learner rows per tick
        SelfPlayTrainer(64, device="cuda:0", opponents=[np.zeros(A_N, np.float32)], pool_envs=64, replay_capacity=256, n_step=5)
    for t in (0, 65, -1):
        with pytest.raises(ValueError, match="tick_rows"):
            ReplayRing(64, device="cpu", tick_rows=t)
    ring = ReplayRing(64, device="cpu")
    ring.advance(40)
    with pytest.raises(ValueError, match="tick_rows"):
        ring.sample(8, n_step=3)
    ring.mark_break()
    assert ring.breaks == []                          # a ring without tick_rows keeps none
    ring = ReplayRing(64, device="cpu", tick_rows=16)
    ring.advance(16)
    with pytest.raises(ValueError, match="no row of the ring"):
        ring.sample(8, n_step=2)
    with pytest.raises(ValueError, match="n_step must be"):
        ring.sample(8, n_step=0)
    with pytest.raises(ValueError, match="at least 80"):
        ring.sample(8, n_step=5)


def test_header_constants_match_the_python_mirror():
    _l = _lib()
    text = open(os.path.join(ROOT, "include", "skillshot_b200.h")).read()
    assert int(re.search(r"#define\s+SS_REPLAY_MAX_RUNS\s+(\d+)", text).group(1)) == _l.REPLAY_MAX_RUNS
    assert int(re.search(r"#define\s+SS_REPLAY_MAX_NSTEP\s+(\d+)", text).group(1)) == _l.REPLAY_MAX_NSTEP
    assert _l.REPLAY_MAX_NSTEP < 256                  # steps_out is one byte


def test_nstep_discount_is_the_float32_recurrence():
    from skillshot_learning_b200.learner import nstep_discount
    g = np.float32(1)
    for n in range(1, 33):
        g = np.float32(g * np.float32(0.99))
        assert nstep_discount(0.99, n) == float(g)
    assert nstep_discount(0.99, 1) == float(np.float32(0.99)) and nstep_discount(0.0, 5) == 0.0


# ---- the agreement of the ranks on n_step (gloo, world size 2, under a timeout) ---------------------------------------
WORLD = 2


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _gloo_case(rank, case):
    import torch.distributed as dist
    from skillshot_learning_b200 import SelfPlayTrainer
    try:
        if case == "differ":           # rank 1 passes another n_step; both are valid
            SelfPlayTrainer(64, device="cpu", process_group=True, n_step=3 + 2 * rank)
        elif case == "refuse":         # rank 1 refuses its n_step
            SelfPlayTrainer(64, device="cpu", process_group=True, n_step=40 if rank == 1 else 3)
        else:                          # both agree: the constructor goes on and fails later, on the CPU device
            SelfPlayTrainer(64, device="cpu", process_group=True, n_step=3)
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


def test_ranks_refuse_a_mismatched_n_step_together(tmp_path):
    m0, m1 = _run("differ", tmp_path)
    assert m0 == m1 == "ValueError: rank 1 passed n_step = 5, rank 0 3"


def test_ranks_raise_together_when_one_refuses_its_n_step(tmp_path):
    m0, m1 = _run("refuse", tmp_path)
    assert m0 == m1 == "ValueError: rank 1 refused: n_step must be an integer in 1..32, got 40"


def test_equal_n_steps_pass_the_agreement(tmp_path):
    m0, m1 = _run("agree", tmp_path)
    assert m0 == m1 and "n_step" not in (m0 or "")


# ---------------------------------------------------------------------------------------------------------------------
# on the GPU
# ---------------------------------------------------------------------------------------------------------------------
gpu = pytest.mark.gpu
DEV = "cuda:0"


def _random_ring(capacity, frames, W, seed, tick_rows=True, fill=None):
    from skillshot_learning_b200 import ReplayRing
    rng = np.random.default_rng(seed)
    ring = ReplayRing(capacity, device=DEV, seed=seed, frames=frames, tick_rows=W if tick_rows else None)
    fill = capacity if fill is None else fill
    for _ in range(fill // W):
        ring.push(rng.uniform(-1, 1, (W, 12 * frames)).astype(np.float32), rng.uniform(-1, 1, (W, 2)).astype(np.float32),
                  rng.uniform(-1, 1, W).astype(np.float32), rng.uniform(-1, 1, (W, 12 * frames)).astype(np.float32),
                  torch.from_numpy((rng.uniform(size=W) < 0.1).astype(np.uint8)))
    return ring


def _sample_nstep(ring, batch, n_step, gamma, runs=None):
    """ss_replay_sample_nstep called directly (runs: the ring's eligible runs by default)"""
    import ctypes
    runs = ring.eligible_runs(n_step) if runs is None else runs
    table = (ctypes.c_int64 * (2 * len(runs)))(*[v for r in runs for v in r])
    w = 12 * ring.frames
    out = dict(obs=torch.empty((batch, w), device=DEV), act=torch.empty((batch, 2), device=DEV), reward=torch.empty(batch, device=DEV),
               next_obs=torch.empty((batch, w), device=DEV), done=torch.empty(batch, dtype=torch.uint8, device=DEV),
               indices=torch.empty(batch, dtype=torch.int64, device=DEV), steps=torch.empty(batch, dtype=torch.uint8, device=DEV))
    rc = _lib().lib.ss_replay_sample_nstep(ring.obs.data_ptr(), ring.act.data_ptr(), ring.reward.data_ptr(), ring.next_obs.data_ptr(),
                                           ring.done.data_ptr(), ring.capacity, ring.frames, ring.tick_rows, n_step, gamma, table,
                                           len(runs), ring.seed, ring.counter, batch, *[out[k].data_ptr() for k in out],
                                           torch.cuda.current_stream().cuda_stream)
    assert rc == 0
    return out


@gpu
@pytest.mark.parametrize("frames", [1, 20])
@pytest.mark.parametrize("with_breaks", [False, True])
def test_one_step_rows_are_the_uniform_sampler_bit_for_bit(frames, with_breaks):
    W = 24
    ring = _random_ring(W * 30, frames, W, seed=frames)
    for _ in range(7):
        ring.push(*(torch.zeros((W, k)) for k in (12 * frames, 2)), torch.zeros(W), torch.zeros((W, 12 * frames)))   # wraps
        if with_breaks:
            ring.mark_break()
    ring.counter = 5
    assert ring.eligible_runs(1) == [(0, ring.size)] and (len(ring.breaks) > 0) == with_breaks
    got = _sample_nstep(ring, 5000, 1, 0.99)
    want = ring.sample(5000)
    for k in ("obs", "act", "reward", "next_obs", "done", "indices"):
        assert torch.equal(got[k], want[k]), k
    assert bool((got["steps"] == 1).all())


def _walk_reference(ring, idx, n, gamma, W):
    """the walk of each drawn row, restated in numpy float32"""
    d, r = ring.done.cpu().numpy(), ring.reward.cpu().numpy()
    cap = ring.capacity
    B = len(idx)
    rew, last, steps = np.zeros(B, np.float32), np.zeros(B, np.int64), np.zeros(B, np.uint8)
    gm = np.float32(gamma)
    for i, src in enumerate(idx):
        row, s, g, k = int(src), r[int(src)], np.float32(1), 1
        while k < n and not d[row]:
            row = (row + W) % cap
            g = np.float32(g * gm)
            s = np.float32(s + np.float32(g * r[row]))
            k += 1
        rew[i], last[i], steps[i] = s, row, k
    return rew, last, steps


def _check_against_numpy(ring, n, gamma, batch=4096):
    runs = ring.eligible_runs(n)
    total = sum(l for _, l in runs)
    j = philox_ref.replay_indices(batch, total, ring.seed, ring.counter)
    starts = np.cumsum([0] + [l for _, l in runs])
    k = np.searchsorted(starts, j, side="right") - 1
    want_idx = np.array([runs[q][0] for q in k]) + (j - starts[k])
    b = ring.sample(batch, n_step=n, gamma=gamma)
    idx = b["indices"].cpu().numpy()
    assert np.array_equal(idx, want_idx)
    rew, last, steps = _walk_reference(ring, idx, n, gamma, ring.tick_rows)
    obs, nxt = ring.obs.cpu().numpy(), ring.next_obs.cpu().numpy()
    assert np.array_equal(b["reward"].cpu().numpy(), rew)
    assert np.array_equal(b["steps"].cpu().numpy(), steps)
    assert np.array_equal(b["obs"].cpu().numpy(), obs[idx]) and np.array_equal(b["act"].cpu().numpy(), ring.act.cpu().numpy()[idx])
    assert np.array_equal(b["next_obs"].cpu().numpy(), nxt[last])
    assert np.array_equal(b["done"].cpu().numpy(), ring.done.cpu().numpy()[last])
    return steps


def _trainer(**kw):
    from skillshot_learning_b200 import SelfPlayTrainer
    base = dict(device=DEV, seed=3, batch_size=512, gamma=0.99, tau=0.005, reward_mode="looking", tick_limit=40)
    base.update(kw)
    return SelfPlayTrainer(base.pop("n_envs", 256), **base)


@gpu
@pytest.mark.parametrize("n", [3, 5])
def test_nstep_rows_match_a_numpy_walk_on_rollout_rings(n):
    from skillshot_learning_b200.learner import A_N
    rng = np.random.default_rng(2)
    # self-play, wrapped ring, a store=False break
    t = _trainer(n_step=n, n_envs=1024, replay_capacity=2048 * 30)
    t.rollout(25)
    t.rollout(2, store=False)
    t.rollout(20)
    assert t.replay.size == t.replay.capacity and t.replay.pos != 0 and len(t.replay.breaks) == 1
    assert int(t.replay.done.sum()) > 0
    steps = _check_against_numpy(t.replay, n, 0.99)
    assert (steps < n).any() and (steps == n).any()              # walks that stopped at a hit and walks of n ticks
    # a pool with a set_pool_blocks break, then rollout_tick(store=False) and record_boards(store=False)
    t = _trainer(n_step=n, opponents=[lo.init_actor(rng), lo.init_actor(rng)], pool_envs=128, replay_capacity=384 * 16)
    t.rollout(5)
    t.set_pool_blocks([96, 32])
    t.rollout(4)
    t.rollout_tick(store=False)
    t.rollout(3)
    t.record_boards(0, 1, store=False)
    t.rollout(2)
    assert len(t.replay.breaks) == 3 and t.replay.size < t.replay.capacity
    _check_against_numpy(t.replay, n, 0.99)
    # the frame-stacked ring (rows of 240 floats), gamma = 0: the reward is the first row's
    t = _trainer(n_step=n, frames=20, n_envs=128, replay_capacity=256 * 10)
    t.rollout(13)
    _check_against_numpy(t.replay, n, 0.0)


@gpu
def test_a_million_draws_cover_exactly_the_eligible_rows_uniformly():
    from scipy.stats import chisquare
    W, n = 16, 4
    ring = _random_ring(W * 300, 1, W, seed=9)
    for _ in range(40):
        ring.push(*(torch.zeros((W, k)) for k in (12, 2)), torch.zeros(W), torch.zeros((W, 12)))
        if _ % 9 == 0:
            ring.mark_break()
    runs = ring.eligible_runs(n)
    eligible = np.zeros(ring.capacity, bool)
    for s, l in runs:
        eligible[s:s + l] = True
    assert 1 < len(runs) and eligible.sum() < ring.size
    counts = np.zeros(ring.capacity, np.int64)
    for _ in range(4):
        b = ring.sample(1 << 18, n_step=n, gamma=0.9)
        counts += np.bincount(b["indices"].cpu().numpy(), minlength=ring.capacity)
    assert counts.sum() == 1 << 20 and counts[~eligible].sum() == 0
    assert chisquare(counts[eligible]).pvalue > 1e-3


def _same_state(a, b):
    na, nb = a.networks, b.networks
    for k in ("params", "target", "adam_m", "adam_v"):
        assert torch.equal(getattr(na, k), getattr(nb, k)), k
    assert (na.step_actor, na.step_critic, na.counter) == (nb.step_actor, nb.step_critic, nb.counter)
    for k in ("obs", "act", "reward", "next_obs", "done"):
        assert torch.equal(getattr(a.replay, k), getattr(b.replay, k)), k
    assert (a.replay.pos, a.replay.size, a.replay.counter) == (b.replay.pos, b.replay.size, b.replay.counter)


@gpu
@pytest.mark.parametrize("path", ["single", "stepwise", "frames", "pool", "td3"])
def test_n_step_one_is_the_default_trainer_bit_for_bit(path, monkeypatch):
    lib = _lib().lib
    calls = []
    real = lib.ss_ddpg_update
    monkeypatch.setattr(lib, "ss_ddpg_update", lambda *a: calls.append(1) or real(*a))
    kw = dict(reward_mode="terminal", precision="bf16")
    if path == "frames":
        kw.update(frames=20, n_envs=128)
    if path == "pool":
        rng = np.random.default_rng(1)
        kw.update(opponents=[lo.init_actor(rng), lo.init_actor(rng, 20)], pool_envs=128)
    if path == "td3":
        kw.update(twin_critics=True, policy_delay=2, target_noise=0.2)
    a, b = _trainer(**kw), _trainer(n_step=1, **kw)
    assert b.replay.tick_rows is None
    for _ in range(20):
        for t in (a, b):
            t.rollout(2)
            t.update_stepwise() if path == "stepwise" else t.update()
    _same_state(a, b)
    assert len(calls) == (40 if path in ("single", "pool") else 0)
    assert set(b.state_dict()["replay"]) == set(a.state_dict()["replay"])


@gpu
@pytest.mark.parametrize("td3", [False, True])
def test_nstep_updates_track_the_oracle(td3):
    """float32, gamma 0.99, tau 0.005, Philox dropout: n-step updates of ActorCritic against TD3Oracle (one critic, no
    smoothing, delay 1 is the DDPG update) given the minibatch the sampler drew and g_n as its gamma."""
    from skillshot_learning_b200 import ActorCritic
    from skillshot_learning_b200.learner import nstep_discount
    rng = np.random.default_rng(4)
    theta, phi = lo.init_actor(rng), lo.init_critic(rng)
    n, W, batch = 4, 32, 96
    opts = dict(twin_critics=True, policy_delay=2) if td3 else {}
    ac = ActorCritic(device=DEV, seed=7, gamma=0.99, tau=0.005, **opts)
    ac.set_weights(theta, phi, **(dict(critic2=ac.critic2.clone()) if td3 else {}))
    g_n = nstep_discount(0.99, n)
    orc = td3_oracle.TD3Oracle(theta, phi, ac.critic2.cpu().numpy() if td3 else None, gamma=g_n, tau=0.005,
                               policy_delay=2 if td3 else 1, sigma=0.0, dropout=0.2)
    ring = _random_ring(W * 40, 1, W, seed=5)
    ring.mark_break()
    ring.push(*(torch.rand((W, k)) for k in (12, 2)), torch.rand(W), torch.rand((W, 12)))
    for _ in range(6):
        k = ac.counter
        if td3:
            b = ring.sample(batch, n_step=n, gamma=0.99)
            ac.td3_step(b["obs"], b["act"], b["reward"], b["next_obs"], b["done"], discount=g_n)
            keeps = [philox_ref.dropout_keep(batch, ac.seed, k + j, 0.2).astype(np.float32) for j in (0, 1)]
        else:
            b = ac.update_from_ring(ring, batch, n_step=n)
            keeps = [philox_ref.dropout_keep(batch, ac.seed, k, 0.2).astype(np.float32), None]
        s, a, r, s2, d = (b[x].cpu().numpy() for x in ("obs", "act", "reward", "next_obs", "done"))
        y = orc.update(s, a, r, s2, d, None, *keeps)
        if not td3:
            np.testing.assert_allclose(b["y"].cpu().numpy(), y, rtol=0, atol=2e-5 * max(1.0, np.abs(y).max()))
    pairs = [(ac.actor, orc.theta), (ac.critic, orc.phi), (ac.target_actor, orc.theta_t), (ac.target_critic, orc.phi_t)]
    if td3:
        pairs += [(ac.critic2, orc.phi2), (ac.target_critic2, orc.phi2_t)]
    for got, want in pairs:
        np.testing.assert_allclose(got.cpu().numpy(), want, rtol=0, atol=2e-5)


@gpu
@pytest.mark.parametrize("cfg", ["single", "pool"])
def test_nstep_checkpoint_resumes_bit_identically(cfg, tmp_path):
    kw = dict(n_step=3, reward_mode="terminal")
    if cfg == "pool":
        rng = np.random.default_rng(1)
        kw.update(opponents=[lo.init_actor(rng), lo.init_actor(rng)], pool_envs=128, precision="bf16", twin_critics=True)
    a = _trainer(**kw)
    a.rollout(6)
    a.rollout(1, store=False)
    if cfg == "pool":
        a.set_pool_blocks([64, 64])
    for _ in range(3):
        a.rollout(2)
        a.update()
    assert a.replay.breaks
    a.save(str(tmp_path / "ck.pt"))
    b = _trainer(**kw)
    b.load(str(tmp_path / "ck.pt"))
    assert b.replay.breaks == a.replay.breaks
    for _ in range(6):
        for t in (a, b):
            t.rollout(2)
            t.update()
    _same_state(a, b)
    assert a.replay.breaks == b.replay.breaks
    # a checkpoint without breaks (an n_step = 1 run) loads with an empty ring
    c = _trainer(**dict(kw, n_step=1))
    c.rollout(4)
    c.save(str(tmp_path / "old.pt"))
    d = _trainer(**kw)
    d.load(str(tmp_path / "old.pt"))
    assert (d.replay.pos, d.replay.size, d.replay.breaks) == (0, 0, [])
    assert torch.equal(d.networks.params, c.networks.params)
    with pytest.raises(ValueError, match="no row of the ring"):
        d.update()
    d.rollout(4)
    d.update()
