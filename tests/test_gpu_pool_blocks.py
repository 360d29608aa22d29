"""Pool blocks of any size per opponent (ss_env_step_pool_blocks, ss_pool_restart, the block table of
ss_pool_rollout_frames, pool_layout(..., blocks), pfsp_blocks and SelfPlayTrainer.set_pool_blocks / rebalance_pool).
The GPU tests compare with ==: the block step against ss_env_step_pool and against ss_env_step_ring under the layout's
permutation, its counters against a host tally, the one-call rollout against its stepwise composition, constant-action
opponents against the C oracle, the restart against an auto-reset tick and ss_env_reset, and the trainer's re-layout and
checkpoints against uninterrupted runs.  The unmarked tests run without a GPU: the host layout, pfsp_blocks and the
rejection of bad block tables."""
import ctypes
import math

import numpy as np
import pytest

from tests.test_gpu_pool import MODES, _crafted_double_hits
from tests.test_gpu_pool_frames import _Setup, _actor, _args, _const_actor, _n_params, _ptr, _same

STRIDE = 36484


def _table(blocks):
    return (ctypes.c_int64 * len(blocks))(*blocks)


# ---------------------------------------------------------------- CPU ------------------------------------------------------------------
@pytest.mark.parametrize("n,blocks", [(64, [32]), (100, [8, 30, 10]), (4096, [2] * 63 + [4096 - 126]), (300, [2, 4, 200, 6, 18])])
def test_block_layout_is_a_seat_balanced_permutation(n, blocks):
    from skillshot_learning_b200.learner import pool_layout
    K, M = len(blocks), sum(blocks)
    S, L = n - M, 2 * n - M
    rows = pool_layout(n, M, K, blocks)
    assert sorted(rows.reshape(-1).tolist()) == list(range(2 * n))
    assert np.array_equal(rows[:S], np.arange(2 * S).reshape(S, 2))
    start = 0
    for b in blocks:
        blk = rows[S + start:S + start + b]
        learner = blk < L
        assert (learner.sum(1) == 1).all()
        assert learner[:b // 2, 0].all() and learner[b // 2:, 1].all()
        assert np.array_equal(np.sort(blk[~learner]), L + np.arange(start, start + b))
        assert np.array_equal(np.sort(blk[learner]), 2 * S + np.arange(start, start + b))
        start += b


@pytest.mark.parametrize("n,M,K", [(64, 32, 1), (100, 48, 3), (4096, 4096, 16), (130, 128, 64)])
def test_uniform_blocks_are_the_uniform_layout(n, M, K):
    from skillshot_learning_b200.learner import pool_layout
    assert np.array_equal(pool_layout(n, M, K, [M // K] * K), pool_layout(n, M, K))


def test_bad_blocks_are_refused_by_the_layout_and_the_trainer():
    from skillshot_learning_b200 import SelfPlayTrainer
    from skillshot_learning_b200.learner import pool_layout
    for blocks in ([16, 16], [16, 15, 17], [0, 24, 24], [16, 16, 18], [1, 23, 24]):
        with pytest.raises(ValueError):
            pool_layout(96, 48, 3, blocks)
        with pytest.raises(ValueError):
            SelfPlayTrainer(96, device="cpu", opponents=[_actor(1)] * 3, pool_envs=48, pool_blocks=blocks)


def test_pfsp_blocks():
    from skillshot_learning_b200.learner import pfsp_blocks
    rng = np.random.default_rng(0)
    for _ in range(300):
        K = int(rng.integers(1, 65))
        m = 2 * int(rng.integers(1, 4))
        M = K * m + 2 * int(rng.integers(0, 3000))
        s = rng.uniform(0, 1, K)
        s[rng.uniform(size=K) < 0.1] = np.nan
        for w in ("hard", "variance", "uniform"):
            out = pfsp_blocks(list(s), M, w, p=float(rng.uniform(0.5, 3)), min_envs=m)
            assert len(out) == K and sum(out) == M and all(b % 2 == 0 and b >= m for b in out)
        out = pfsp_blocks(list(s), M, "hard", 2.0, m)
        t = np.where(np.isnan(s), 0.5, s)
        for a in range(K):
            for b in range(K):
                if t[a] < t[b]:
                    assert out[a] >= out[b]                    # a lower score never gets fewer envs
    assert pfsp_blocks([0.3] * 8, 1024) == [128] * 8 == pfsp_blocks([0.9] * 8, 1024, "variance")
    assert pfsp_blocks([None, float("nan"), 0.5], 96) == [32] * 3
    assert pfsp_blocks([1.0, 1.0], 40) == [20, 20]                       # every weight 0: the uniform split
    assert pfsp_blocks([0.0, 1.0], 40) == [38, 2]
    # fixed inputs, fixed outputs (largest remainder, ties to the lower k)
    # weights .01 .25 .81 .09 over 96 units: quotas .83 20.69 67.03 7.45, the two units left to k = 0 and 1
    assert pfsp_blocks([0.9, 0.5, 0.1, 0.7], 200) == [4, 44, 136, 16]
    assert pfsp_blocks([0.5, 0.5, 0.5], 32) == [12, 10, 10]
    for args in (([0.5] * 3, 30, "soft"), ([0.5] * 3, 31), ([0.5] * 3, 4), ([1.5], 8), ([-0.1], 8), ([], 8), ([0.5] * 65, 1000),
                 ([0.5] * 2, 40, "hard", -1.0), ([0.5] * 2, 40, "hard", math.inf), ([0.5] * 2, 40, "hard", 2.0, 3),
                 ([0.5] * 2, 40, "hard", 2.0, 0)):
        with pytest.raises(ValueError):
            pfsp_blocks(*args)


def test_bad_block_tables_are_rejected_without_a_gpu():
    from skillshot_learning_b200 import _lib
    L, P = _lib.lib, 4096
    bad = ([16, 16, 18], [16, 15, 17], [0, 24, 24], [1, 23, 24], [16, 16, 14])

    def step(table, M=48):
        return L.ss_env_step_pool_blocks(P, 96, M, 3, P, P, P, None, P, None, P, None, None, 1, 100, 1, 0, 0, None, 0, None, table, None)
    for blocks in bad:
        t = _table(blocks)
        assert step(t) == -1, blocks
        assert L.ss_pool_restart(P, 96, 48, 3, t, 1, 0, 0, P, P, None, None) == -1, blocks
        a = _args(opp_envs=t)
        assert L.ss_pool_rollout_frames(ctypes.byref(a), None) == -1, blocks
        assert L.ss_pool_rollout_frames_workspace_bytes(ctypes.byref(a)) == -1, blocks
    assert step(_table([16, 16, 16]), M=0) == -1                        # no pool envs take no table
    assert L.ss_pool_restart(P, 96, 48, 3, None, 2, 0, 0, P, P, None, None) == -1
    assert L.ss_pool_restart(P, 96, 0, 3, None, 1, 0, 0, P, P, None, None) == -1
    assert L.ss_pool_restart(P, 96, 45, 3, None, 1, 0, 0, P, P, None, None) == -1
    # the workspace: the largest layer-1 scratch of the learner and of the 20-frame opponent's block
    for blocks in ([16, 16, 16], [2, 40, 6], [30, 2, 16]):
        need = L.ss_pool_rollout_frames_workspace_bytes(ctypes.byref(_args(opp_envs=_table(blocks))))
        assert need == 2 * 45700 * 4 + max(L.ss_actor_frames_tc_workspace_bytes(144, 128), L.ss_actor_frames_tc_workspace_bytes(blocks[1], 0))
    assert L.ss_pool_rollout_frames_workspace_bytes(ctypes.byref(_args(opp_envs=_table([16, 16, 16])))) == \
        L.ss_pool_rollout_frames_workspace_bytes(ctypes.byref(_args()))


# ---------------------------------------------------------------- GPU: the step ---------------------------------------------------------
class _Steps:
    """The same envs stepped by ss_env_step_ring ([n][2] rows), by ss_env_step_pool_blocks under `blocks` and, for uniform
    blocks, by ss_env_step_pool."""

    def __init__(self, n, blocks, mode="looking", random_positions=True, tick_limit=40, seed=3):
        import torch
        from skillshot_learning_b200 import SkillshotEnvs
        from skillshot_learning_b200.learner import pool_layout
        K, M = len(blocks), sum(blocks)
        self.n, self.M, self.K, self.L, self.blocks = n, M, K, 2 * n - M, list(blocks)
        self.uniform = blocks == [M // K] * K
        self.mode, self.limit, self.seed, self.reset = MODES[mode], tick_limit, seed, 1 if random_positions else 0
        self.env = SkillshotEnvs(n, random_positions=random_positions, seed=seed)
        self.states = dict(ring=self.env.state.clone(), blocks=self.env.state.clone(), pool=self.env.state.clone())
        self.rows = torch.from_numpy(pool_layout(n, M, K, blocks).reshape(-1)).cuda()
        d = dict(device="cuda")
        self.out = dict(ring=dict(obs=torch.zeros(2 * n, 12, **d), obs2=torch.zeros(2 * n, 12, **d), reward=torch.zeros(2 * n, **d),
                                  done=torch.zeros(n, dtype=torch.uint8, **d), done_rows=torch.zeros(2 * n, dtype=torch.uint8, **d),
                                  winner=torch.zeros(n, dtype=torch.uint8, **d), status=torch.zeros(2 + 144, dtype=torch.int32, **d)))
        for k in ("blocks", "pool"):
            self.out[k] = dict(obs=torch.zeros(self.L, 12, **d), obs2=torch.zeros(self.L, 12, **d), reward=torch.zeros(self.L, **d),
                               done=torch.zeros(n, dtype=torch.uint8, **d), done_rows=torch.zeros(self.L, dtype=torch.uint8, **d),
                               winner=torch.zeros(n, dtype=torch.uint8, **d), status=torch.zeros(2 + 144, dtype=torch.int32, **d),
                               opp_obs=torch.zeros(M, 12, **d), stats=torch.zeros(K, 8, dtype=torch.int64, **d))
        self.table = _table(blocks)
        self.counter = 100

    def tick(self, act):
        import torch
        from skillshot_learning_b200._lib import lib
        R = self.out["ring"]
        assert lib.ss_env_step_ring(self.states["ring"].data_ptr(), self.n, act.data_ptr(), R["obs"].data_ptr(), R["obs2"].data_ptr(),
                                    R["reward"].data_ptr(), R["done"].data_ptr(), R["done_rows"].data_ptr(), R["winner"].data_ptr(), 1,
                                    self.mode, self.limit, 1, self.reset, self.seed, self.counter, None, R["status"].data_ptr(), 2,
                                    None) == 0
        comb = torch.empty(2 * self.n, 2, device="cuda")
        comb[self.rows] = act.reshape(-1, 2)
        la, oa = comb[:self.L].contiguous(), comb[self.L:].contiguous()
        for k, fn in (("blocks", lib.ss_env_step_pool_blocks), ("pool", lib.ss_env_step_pool)):
            if k == "pool" and not self.uniform:
                continue
            Q = self.out[k]
            args = [self.states[k].data_ptr(), self.n, self.M, self.K, la.data_ptr(), oa.data_ptr(), Q["obs"].data_ptr(), Q["obs2"].data_ptr(),
                    Q["reward"].data_ptr(), Q["done_rows"].data_ptr(), Q["opp_obs"].data_ptr(), Q["done"].data_ptr(), Q["winner"].data_ptr(),
                    self.mode, self.limit, self.reset, self.seed, self.counter, Q["status"].data_ptr(), 2, Q["stats"].data_ptr()]
            assert fn(*(args + ([self.table] if k == "blocks" else []) + [None])) == 0
        self.counter += 1
        torch.cuda.synchronize()
        Q = self.out["blocks"]
        assert torch.equal(self.states["ring"], self.states["blocks"])
        assert torch.equal(R["done"], Q["done"]) and torch.equal(R["winner"], Q["winner"]) and torch.equal(R["status"], Q["status"])
        obs = torch.cat([Q["obs"], Q["opp_obs"]])[self.rows]
        assert torch.equal(obs, R["obs"]) and torch.equal(Q["obs2"], Q["obs"])
        learner = self.rows < self.L
        lr = self.rows[learner]
        assert torch.equal(Q["done_rows"][lr], R["done_rows"][learner])
        if self.mode:
            assert torch.equal(Q["reward"][lr], R["reward"][learner])
        if self.uniform:
            assert torch.equal(self.states["pool"], self.states["blocks"])
            for k, v in self.out["pool"].items():
                assert torch.equal(v, Q[k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 3, 16])
def test_uniform_block_step_is_the_pool_step(K):
    import torch
    n, M = 2000 + 96 * K, 96 * K
    s = _Steps(n, [M // K] * K, mode="looking", tick_limit=25)
    g = torch.Generator(device="cuda").manual_seed(K)
    for _ in range(60):
        s.tick(torch.rand(n, 2, 2, device="cuda", generator=g) * 2.4 - 1.2)
    assert s.out["pool"]["stats"][:, 0].sum() > 0


def _blocks(K, seed):
    """K unequal even blocks >= 2: sizes 2 .. 2 + 2 * 40"""
    rng = np.random.default_rng(seed)
    return [2 + 2 * int(v) for v in rng.integers(0, 41, K)]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["none", "looking", "terminal"])
@pytest.mark.parametrize("K", [1, 3, 16, 64])
def test_block_step_is_the_ring_step_under_the_layout(K, mode):
    import torch
    blocks = _blocks(K, K)
    n = 1500 + sum(blocks)
    s = _Steps(n, blocks, mode=mode, random_positions=K % 2 == 1, tick_limit=25)
    g = torch.Generator(device="cuda").manual_seed(K)
    for _ in range(60):                                  # several auto-resets at the tick limit
        s.tick(torch.rand(n, 2, 2, device="cuda", generator=g) * 2.4 - 1.2)
    assert s.out["blocks"]["stats"][:, 0].sum() > 0


@pytest.mark.gpu
def test_block_counters_equal_a_host_tally():
    import torch
    blocks = [8, 200, 12, 340, 400]
    n, M, K = 1200, sum(blocks), len(blocks)
    S = n - M
    starts = np.concatenate([[0], np.cumsum(blocks)])
    s = _Steps(n, blocks, mode="terminal", random_positions=False, tick_limit=30)
    crafted = [S + int(starts[k]) + q for k in range(K) for q in (0, 3, blocks[k] - 1, blocks[k] - 4)]   # the learner in both seats
    env = s.env
    env.state.copy_(s.states["ring"])
    _crafted_double_hits(env, crafted)
    for st in s.states.values():
        st.copy_(env.state)
    length = env.export_state()["ticks"].astype(np.int64)
    tally = np.zeros((K, 8), np.int64)
    g = torch.Generator(device="cuda").manual_seed(7)
    doubles = 0
    for t in range(80):
        act = torch.rand(n, 2, 2, device="cuda", generator=g) * 2.4 - 1.2
        if t == 0:
            act[crafted] = 0.0
        s.tick(act)
        done, winner = s.out["blocks"]["done"].cpu().numpy(), s.out["blocks"]["winner"].cpu().numpy()
        length += 1
        for j in np.nonzero(done[S:])[0]:
            k = int(np.searchsorted(starts, j, side="right") - 1)
            lp = int(j - starts[k] >= blocks[k] // 2)
            c = tally[k]
            c[0] += 1
            w = int(winner[S + j])
            c[3 if w == 0 else 2 if w == lp + 1 else 1] += 1
            c[4] += length[S + j]
            if t == 0 and S + j in crafted:
                doubles += 1
        length[done != 0] = 0
    assert doubles == len(crafted)
    assert tally[:, 1].sum() > 0 and tally[:, 2].sum() > 0 and tally[:, 3].sum() > 0
    assert np.array_equal(s.out["blocks"]["stats"].cpu().numpy(), tally)


@pytest.mark.gpu
@pytest.mark.parametrize("random_positions", [False, True])
def test_restart_is_an_auto_reset_and_an_env_reset(random_positions):
    """ss_pool_restart with counter c gives the state and observations of a tick with counter c that ends (and so
    auto-resets) every game, and the state of ss_env_reset over the pool envs; the self-play envs are untouched."""
    import torch
    from skillshot_learning_b200._lib import lib
    blocks = [6, 40, 2, 18, 30]
    n, M, K = 700, sum(blocks), len(blocks)
    S, L = n - M, 2 * n - M
    s = _Steps(n, blocks, mode="looking", random_positions=random_positions, tick_limit=1)
    g = torch.Generator(device="cuda").manual_seed(4)
    for _ in range(3):                                   # (games of any state: every tick ends and restarts all of them)
        s.tick(torch.rand(n, 2, 2, device="cuda", generator=g) * 2.4 - 1.2)
    start = s.states["blocks"].clone()
    obs, opp = torch.full((L, 12), -7.0, device="cuda"), torch.full((M, 12), -7.0, device="cuda")
    obs0 = obs.clone()
    c, reset = s.counter, 1 if random_positions else 0
    assert lib.ss_pool_restart(start.data_ptr(), n, M, K, s.table, reset, s.seed, c, obs.data_ptr(), opp.data_ptr(), None, None) == 0
    s.tick(torch.rand(n, 2, 2, device="cuda", generator=g) * 2.4 - 1.2)       # every game ends under counter c
    ref = s.env
    ref.state.copy_(s.states["ring"])
    torch.cuda.synchronize()
    mine = {k: v.copy() for k, v in _export(ref, start).items()}
    tick = _export(ref, s.states["blocks"])
    for k in mine:
        assert np.array_equal(mine[k][S:], tick[k][S:]), k
    Q = s.out["blocks"]
    assert torch.equal(obs[2 * S:], Q["obs"][2 * S:]) and torch.equal(opp, Q["opp_obs"])
    assert torch.equal(obs[:2 * S], obs0[:2 * S])
    # against ss_env_reset of the pool envs; the self-play envs are as they were
    before = s.states["ring"].clone()
    ref.state.copy_(before)
    mask = torch.zeros(n, dtype=torch.uint8, device="cuda")
    mask[S:] = 1
    assert lib.ss_env_reset(ref.state.data_ptr(), n, mask.data_ptr(), reset, None, s.seed, c + 1, None) == 0
    again = before.clone()
    assert lib.ss_pool_restart(again.data_ptr(), n, M, K, s.table, reset, s.seed, c + 1, obs.data_ptr(), opp.data_ptr(), None, None) == 0
    torch.cuda.synchronize()
    assert torch.equal(again, ref.state)


def _export(env, state):
    keep = env.state.clone()
    env.state.copy_(state)
    out = env.export_state()
    env.state.copy_(keep)
    return out


# ---------------------------------------------------------------- GPU: the rollout -----------------------------------------------------
class _BlockSetup(_Setup):
    """_Setup under a block table: observations in the block layout, each opponent's history at its b_k rows."""

    def __init__(self, n, blocks, frames, opp_frames, precision, segs, table=True, seed=5):
        import torch
        from skillshot_learning_b200._lib import lib
        from skillshot_learning_b200.learner import pool_layout
        M, K = sum(blocks), len(blocks)
        super().__init__(n, M, frames, [1] * K, precision, segs, seed)       # (histories of the opponents below)
        self.blocks, self.starts, self.opp_frames = list(blocks), [0] + list(np.cumsum(blocks)), list(opp_frames)
        self.use_table = table
        self.stride = max((_n_params(f) + 3) // 4 * 4 for f in opp_frames)
        self.opp = torch.zeros(K, self.stride, device="cuda")
        for k, f in enumerate(opp_frames):
            self.opp[k, :_n_params(f)] = _actor(40 + k, frames=f, scale=4.0).cuda()
        rows = torch.from_numpy(pool_layout(n, M, K, blocks).reshape(-1)).cuda()
        self.obs[rows] = self.env.observe().reshape(-1, 12)
        self.restart_histories()

    def restart_histories(self):
        import torch
        from skillshot_learning_b200._lib import lib
        L, n, M = self.L, self.n, self.M
        ones = torch.ones(n, dtype=torch.uint8, device="cuda")
        if self.F > 1:
            assert lib.ss_obs_stack_push_pool(_ptr(self.stack_tc), self.stack32.data_ptr(), n, M, self.F, self.head, self.obs.data_ptr(),
                                              ones.data_ptr(), self.rows.data_ptr(), None, None) == 0
        self.opp_stacks = []
        for k, (f, b) in enumerate(zip(self.opp_frames, self.blocks)):
            if f == 1:
                self.opp_stacks.append(None)
                continue
            s = torch.zeros(lib.ss_obs_stack_tc_bytes(b, f), dtype=torch.uint8, device="cuda") if self.tc else torch.zeros(b, f, 12, device="cuda")
            push = lib.ss_obs_stack_push_tc if self.tc else lib.ss_obs_stack_push
            assert push(s.data_ptr(), b, f, self.head, self.obs[L + self.starts[k]:].data_ptr(), None, 1, None) == 0
            self.opp_stacks.append(s)

    def args(self, n_ticks, write_pos, env_counter, noise_counter):
        import torch
        from skillshot_learning_b200 import _lib
        L, r = self.L, self.ring
        a = _lib.PoolRolloutFramesArgs()
        a.state, a.n_envs, a.pool_envs, a.n_opponents = self.env.state.data_ptr(), self.n, self.M, self.K
        a.params, a.opp_params, a.opp_param_stride = self.params.data_ptr(), self.opp.data_ptr(), self.stride
        a.obs, a.act, a.reward = self.obs.data_ptr(), self.act.data_ptr(), self.reward.data_ptr()
        a.opp_obs, a.opp_act = self.obs[L:].data_ptr(), self.act[L:].data_ptr()
        a.done, a.winner = self.done.data_ptr(), self.winner.data_ptr()
        a.ring_obs, a.ring_act, a.ring_reward, a.ring_next_obs, a.ring_done = (r[k].data_ptr() for k in ("obs", "act", "reward", "next_obs", "done"))
        a.capacity, a.write_pos, a.n_ticks = self.cap, write_pos, n_ticks
        a.param_noise_sd, a.noise_group, a.tensor_cores, a.reward_mode, a.tick_limit = 0.5, 128, self.tc, 1, 60
        a.reset_mode, a.env_seed, a.env_counter, a.noise_seed, a.noise_counter = 1, 5, env_counter, 11, noise_counter
        a.status, a.step_flags, a.pool_stats = self.status.data_ptr(), 2, self.stats.data_ptr()
        a.frames, a.stack_tc, a.stack32, a.rows, a.head = self.F, _ptr(self.stack_tc), _ptr(self.stack32), _ptr(self.rows), self.head
        a._keep = ((ctypes.c_int * self.K)(*self.opp_frames), (ctypes.c_void_p * self.K)(*[_ptr(s) for s in self.opp_stacks]),
                   _table(self.blocks) if self.use_table else None)
        a.opp_frames, a.opp_stacks, a.opp_envs = a._keep
        need = _lib.lib.ss_pool_rollout_frames_workspace_bytes(ctypes.byref(a))
        assert need >= 0
        if need:
            self.ws = torch.zeros(need, dtype=torch.uint8, device="cuda")
            a.workspace, a.workspace_bytes = self.ws.data_ptr(), need
        return a

    def stepwise(self, n_ticks, write_pos, env_counter, noise_counter):
        """ss_pool_rollout_frames with a block table composed from the existing entry points, tick by tick"""
        import torch
        from skillshot_learning_b200._lib import lib
        from tests.test_gpu_pool_frames import _env_of_row
        n, M, K, L, F, r = self.n, self.M, self.K, self.L, self.F, self.ring
        B, st = self.blocks, self.starts
        segs, seg = self.cap // L, write_pos // L
        r["obs"][seg * L:(seg + 1) * L] = self.rows if F > 1 else self.obs[:L]
        env = torch.from_numpy(_env_of_row(n, M)).cuda()
        stride = (_n_params(F) + 3) // 4 * 4
        groups = (L + 127) // 128
        noisy = torch.zeros(groups * stride, device="cuda")
        ws = torch.zeros(max([lib.ss_actor_frames_tc_workspace_bytes(L, 128)] + [lib.ss_actor_frames_tc_workspace_bytes(b, 0) for b in B]),
                         dtype=torch.uint8, device="cuda")
        oo, oa = self.obs[L:], self.act[L:]
        table = _table(B)
        for t in range(n_ticks):
            head, last, nxt = self.head + t, t + 1 == n_ticks, (seg + 1) % segs
            o, a = r["obs"][seg * L:(seg + 1) * L], r["act"][seg * L:(seg + 1) * L]
            if F > 1:
                assert lib.ss_param_noise_groups(self.params.data_ptr(), noisy.data_ptr(), _n_params(F), groups, stride, 0.5, 11,
                                                 noise_counter + t, None) == 0
                fwd = lib.ss_actor_forward_frames_tc if self.tc else lib.ss_actor_forward_frames
                extra = [ws.data_ptr(), ws.numel()] if self.tc else []
                hist = self.stack_tc if self.tc else self.stack32
                assert fwd(*([noisy.data_ptr(), stride, 128, hist.data_ptr(), F, head, a.data_ptr(), L] + extra + [None])) == 0
            else:
                fwd = lib.ss_actor_forward_tc if self.tc else lib.ss_actor_forward
                assert fwd(self.params.data_ptr(), o.data_ptr(), a.data_ptr(), L, 0.5, 128, 0.0, 11, noise_counter + t, None) == 0
            for k, f in enumerate(self.opp_frames):              # (one launch per opponent: the rows are the same)
                p, b, s0 = self.opp[k].data_ptr(), B[k], st[k]
                if f > 1:
                    fwd = lib.ss_actor_forward_frames_tc if self.tc else lib.ss_actor_forward_frames
                    extra = [ws.data_ptr(), ws.numel()] if self.tc else []
                    assert fwd(*([p, 0, 0, self.opp_stacks[k].data_ptr(), f, head, oa[s0:].data_ptr(), b] + extra + [None])) == 0
                elif self.tc:
                    one = (ctypes.c_int64 * 1)(b)
                    assert lib.ss_actor_forward_segments_tc(p, self.stride, one, 1, oo[s0:].data_ptr(), oa[s0:].data_ptr(), None) == 0
                else:
                    assert lib.ss_actor_forward(p, oo[s0:].data_ptr(), oa[s0:].data_ptr(), b, 0.0, 1, 0.0, 0, 0, None) == 0
            if F > 1:
                obs_out, obs2 = self.obs[:L], None
            else:
                obs_out, obs2 = r["next_obs"][seg * L:(seg + 1) * L], (r["obs"][nxt * L:(nxt + 1) * L] if not last else self.obs[:L])
            assert lib.ss_env_step_pool_blocks(self.env.state.data_ptr(), n, M, K, a.data_ptr(), oa.data_ptr(), obs_out.data_ptr(),
                                               _ptr(obs2), r["reward"][seg * L:].data_ptr(), r["done"][seg * L:].data_ptr(), oo.data_ptr(),
                                               self.done.data_ptr(), self.winner.data_ptr(), 1, 60, 1, 5, env_counter + t,
                                               self.status.data_ptr(), 2, self.stats.data_ptr(), table, None) == 0
            if F > 1:
                done_rows = self.done[env].contiguous()
                if self.tc:
                    assert lib.ss_obs_stack_push_tc(self.stack_tc.data_ptr(), L, F, head + 1, self.obs.data_ptr(), done_rows.data_ptr(), 1,
                                                    None) == 0
                assert lib.ss_obs_stack_push(self.stack32.data_ptr(), L, F, head + 1, self.obs.data_ptr(), done_rows.data_ptr(), 1, None) == 0
                assert lib.ss_obs_stack_ordered(self.stack32.data_ptr(), L, F, head + 1, self.rows.data_ptr(), None) == 0
                r["next_obs"][seg * L:(seg + 1) * L] = self.rows
                if not last:
                    r["obs"][nxt * L:(nxt + 1) * L] = self.rows
            for k, f in enumerate(self.opp_frames):
                if f > 1:
                    push = lib.ss_obs_stack_push_tc if self.tc else lib.ss_obs_stack_push
                    assert push(self.opp_stacks[k].data_ptr(), B[k], f, head + 1, oo[st[k]:].data_ptr(), self.done[self.S + st[k]:].data_ptr(),
                                1, None) == 0
            seg = nxt
        last = (seg + segs - 1) % segs
        self.act[:L] = r["act"][last * L:(last + 1) * L]
        self.reward.copy_(r["reward"][last * L:(last + 1) * L])
        self.head += n_ticks
        torch.cuda.synchronize()


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["bf16", "f32"])
@pytest.mark.parametrize("frames,blocks,opp_frames", [(1, [40, 300, 8, 100], [1, 1, 20, 1]), (20, [300, 2, 62], [20, 1, 4]),
                                                      (20, [128, 256], [20, 20]), (1, [2, 510], [20, 1])])
def test_block_rollout_equals_its_stepwise_composition(precision, frames, blocks, opp_frames):
    one = _BlockSetup(1500, blocks, frames, opp_frames, precision, 3)
    two = _BlockSetup(1500, blocks, frames, opp_frames, precision, 3)
    L = one.L
    pos, ec, nc = L, 7, 13
    for rep in range(2):                                  # the ring wraps (3 segments, 2 x 5 ticks from segment 1)
        one.run(5, pos, ec, nc)
        two.stepwise(5, pos, ec, nc)
        _same(one, two)
        pos, ec, nc = (pos + 5 * L) % one.cap, ec + 5, nc + 5
    assert one.stats[:, 0].sum() > 0


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["bf16", "f32"])
def test_uniform_table_is_the_null_table(precision):
    blocks, opp_frames = [96] * 4, [1, 20, 1, 4]
    one = _BlockSetup(1500, blocks, 4, opp_frames, precision, 3, table=True)
    two = _BlockSetup(1500, blocks, 4, opp_frames, precision, 3, table=False)
    for rep in range(2):
        one.run(6, one.L * rep, 7 + 6 * rep, 13 + 6 * rep)
        two.run(6, two.L * rep, 7 + 6 * rep, 13 + 6 * rep)
        _same(one, two)


@pytest.mark.gpu
def test_constant_action_opponents_on_unequal_blocks_equal_the_oracle():
    import torch
    from oracle.oracle import OracleEnvs
    from skillshot_learning_b200._lib import lib
    from skillshot_learning_b200.learner import pool_layout
    n, T = 800, 40
    blocks = [64, 300, 148]
    consts = [((0.898, -0.08), 20), ((0.189, -0.324), 1), ((-0.5, 0.7), 4)]
    s = _BlockSetup(n, blocks, 4, [f for _, f in consts], "bf16", T + 1)
    L, S, K, M = s.L, s.S, len(blocks), sum(blocks)
    s.env.reset(random_positions=False)
    lay = pool_layout(n, M, K, blocks)
    s.obs[torch.from_numpy(lay.reshape(-1)).cuda()] = s.env.observe().reshape(-1, 12)
    s.restart_histories()
    for k, (c, f) in enumerate(consts):
        s.opp[k].zero_()
        s.opp[k, :_n_params(f)] = _const_actor(c, f).cuda()
    a = s.args(T, 0, 0, 0)
    a.reward_mode, a.reset_mode, a.tick_limit = 2, 0, 25
    assert lib.ss_pool_rollout_frames(ctypes.byref(a), None) == 0
    torch.cuda.synchronize()
    opp_act = s.act[L:].cpu().numpy()
    assert all((opp_act[s.starts[k]:s.starts[k + 1]] == opp_act[s.starts[k]]).all() for k in range(K))
    ring = {k: v.cpu().numpy() for k, v in s.ring.items()}
    learner = lay < L
    orc = OracleEnvs(n)
    for t in range(T):
        act = np.empty((n, 2, 2), np.float32)
        act[learner] = ring["act"][t * L + lay[learner]]
        act[~learner] = opp_act[lay[~learner] - L]
        out = orc.step(act, want_obs=False, reward_mode=2, tick_limit=25, auto_reset=True)
        assert out["errors"] == 0
        assert np.array_equal(ring["reward"][t * L + lay[learner]], out["reward"][learner])
        hit = np.repeat((out["winner"] != 0)[:, None], 2, 1)
        assert np.array_equal(ring["done"][t * L + lay[learner]], hit[learner].astype(np.uint8))
    want, got = orc.snapshot(), s.env.export_state()
    for k in ("px", "py", "qx", "qy", "ticks", "live", "winner"):
        assert np.array_equal(got[k], want[k]), k
    assert s.stats[:, 0].sum() > 0 and S > 0


# ---------------------------------------------------------------- GPU: the trainer -----------------------------------------------------
def _mixed(**kw):
    from skillshot_learning_b200 import SelfPlayTrainer
    args = dict(seed=3, batch_size=1024, precision="bf16", tick_limit=40, frames=4,
                opponents=[_actor(20, scale=4.0), _actor(21, frames=20, scale=4.0), _actor(22, frames=4, scale=4.0)])
    args.update(kw)
    return SelfPlayTrainer(1024, **args)


def _tc_rows(stack, n_rows, frames):
    """the fp16 history of ss_obs_stack_push_tc as int16 [n_rows][frames * 12] (slot-major)"""
    import torch
    tiles = (n_rows + 127) // 128
    x = stack.view(torch.float16).view(tiles, -1, 128, 8).permute(0, 2, 1, 3).reshape(tiles * 128, -1)
    return x[:n_rows, :frames * 12].contiguous()


NEW = [300, 110, 100]


@pytest.mark.gpu
def test_set_pool_blocks_restarts_every_pool_game():
    import torch
    from skillshot_learning_b200._lib import lib
    from skillshot_learning_b200.learner import pool_layout
    tr = _mixed()
    assert tr.pool_blocks == [170] * 3
    tr.rollout(5)
    tr.update()
    tr.rollout(3)
    torch.cuda.synchronize()
    n, M, K, L, F = 1024, tr.pool_envs, 3, tr.learner_rows, tr.frames
    S = n - M
    before = dict(state=tr.envs.state.clone(), rows=tr.rows.clone(), s32=tr.stack.stack32.clone(), tc=_tc_rows(tr.stack.stack, L, F).clone(),
                  status=tr.envs.status.clone(), stats=tr.pool_stats.clone(), counter=tr.envs.counter, head=tr.pool_head,
                  ring={k: getattr(tr.replay, k).clone() for k in ("obs", "act", "reward", "next_obs", "done")}, pos=tr.replay.pos)
    tr.set_pool_blocks(NEW)
    torch.cuda.synchronize()
    assert tr.pool_blocks == NEW and tr.envs.counter == before["counter"] + 1 and tr.pool_head == before["head"]
    # the state: ss_env_reset of the pool envs under Philox counter envs.counter
    want = before["state"].clone()
    mask = torch.zeros(n, dtype=torch.uint8, device="cuda")
    mask[S:] = 1
    assert lib.ss_env_reset(want.data_ptr(), n, mask.data_ptr(), 1, None, tr.envs.seed, before["counter"], None) == 0
    torch.cuda.synchronize()
    assert torch.equal(tr.envs.state, want)
    # the self-play rows and histories are byte-identical; every slot of a pool row holds the new game's first observation
    assert torch.equal(tr.rows[:2 * S], before["rows"][:2 * S]) and torch.equal(tr.stack.stack32[:2 * S], before["s32"][:2 * S])
    tc = _tc_rows(tr.stack.stack, L, F)
    assert torch.equal(tc[:2 * S].view(torch.int16), before["tc"][:2 * S].view(torch.int16))
    first = tr.obs[2 * S:L]
    assert torch.equal(tr.stack.stack32[2 * S:], first[:, None, :].expand(-1, F, -1))
    assert torch.equal(tr.rows[2 * S:], first.repeat(1, F))
    assert torch.equal(tc[2 * S:].view(-1, F, 12), first.half()[:, None, :].expand(-1, F, -1))
    lay = torch.from_numpy(pool_layout(n, M, K, NEW).reshape(-1)).cuda()
    np.testing.assert_allclose(tr.obs[lay].cpu().numpy()[2 * S:], tr.envs.observe().reshape(-1, 12).cpu().numpy()[2 * S:], rtol=1e-6,
                               atol=1e-12)
    # the opponents' histories: the new block sizes, filled with their rows' first observation
    start = np.concatenate([[0], np.cumsum(NEW)])
    for k, f in enumerate(tr.opp_frames):
        if f == 1:
            assert tr.opp_stacks[k] is None
            continue
        assert tr.opp_stacks[k].numel() == lib.ss_obs_stack_tc_bytes(NEW[k], f)
        o = tr.obs[L + start[k]:L + start[k + 1]]
        assert torch.equal(_tc_rows(tr.opp_stacks[k], NEW[k], f).view(-1, f, 12), o.half()[:, None, :].expand(-1, f, -1))
    # nothing counted, the ring untouched; the next rollout's first transition starts from the new observations
    assert torch.equal(tr.envs.status, before["status"]) and torch.equal(tr.pool_stats, before["stats"])
    for k, v in before["ring"].items():
        assert torch.equal(getattr(tr.replay, k), v), k
    rows = tr.rows.clone()
    p = tr.replay.pos
    tr.rollout_tick()
    torch.cuda.synchronize()
    assert torch.equal(tr.replay.obs[p:p + L], rows)


def _same_pool(t1, t2):
    import torch
    from tests.test_gpu_pool_frames import _same_pool as same
    same(t1, t2)
    assert t1.pool_blocks == t2.pool_blocks


@pytest.mark.gpu
def test_checkpoint_after_a_relayout_resumes_bit_identically():
    import torch
    t1 = _mixed()
    t1.rollout(3)
    t1.update()
    sd0 = t1.state_dict()
    t1.set_pool_blocks(NEW)
    t1.rollout(3)
    t1.update()
    torch.cuda.synchronize()
    sd = t1.state_dict()
    for _ in range(2):
        t1.rollout(3)
        t1.update()
    t2 = _mixed(seed=8, opponents=[_actor(50), _actor(51, frames=20), _actor(52, frames=4)])
    t2.load_state_dict(sd)
    assert t2.pool_blocks == NEW
    for _ in range(2):
        t2.rollout(3)
        t2.update()
    _same_pool(t1, t2)
    # a checkpoint without blocks loads as uniform, whatever the trainer's layout was
    del sd0["pool"]["blocks"]
    u1, u2 = _mixed(), _mixed(pool_blocks=NEW)
    u1.load_state_dict(sd0)
    u2.load_state_dict(sd0)
    assert u2.pool_blocks == [170] * 3
    for u in (u1, u2):
        u.rollout(4)
        u.update()
    _same_pool(u1, u2)


@pytest.mark.gpu
def test_rebalance_pool_sizes_blocks_by_score():
    import torch
    from skillshot_learning_b200.learner import pfsp_blocks
    tr = _mixed(frames=1)
    tr.rollout(2)
    stats = torch.zeros(3, 8, dtype=torch.int64)
    stats[0, :5] = torch.tensor([100, 90, 5, 5, 3000])           # episodes, wins, losses, draws, ticks
    stats[1, :5] = torch.tensor([40, 10, 20, 10, 800])
    tr.pool_stats.copy_(stats.cuda())
    want = pfsp_blocks([92.5 / 100, 15 / 40, None], tr.pool_envs, "hard", 1.5, 4)
    assert tr.rebalance_pool(p=1.5, min_envs=4) == want == tr.pool_blocks
    assert int(tr.pool_stats.abs().sum()) == 0
    assert want[1] > want[2] > want[0]
