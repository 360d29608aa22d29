"""Training against a pool of frozen opponents (ss_env_step_pool, ss_pool_rollout, SelfPlayTrainer(opponents=...)).
The GPU tests compare with ==: the pool step against ss_env_step_ring under the pool layout's permutation, the pool
counters against a host tally, the one-call rollout against its stepwise composition and (with no pool envs) against
ss_selfplay_rollout, constant-action opponents against the C oracle, and the trainer's checkpoint, set_opponent and
evaluate_league against uninterrupted runs.  The unmarked tests run without a GPU: argument rejection, the argument
block's field order and the host layout."""
import ctypes
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
A_N = 36482
STRIDE = 36484
MODES = {"none": 0, "looking": 1, "terminal": 2}


def _actor(seed, scale=1.0):
    import torch
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(A_N, generator=g) * 0.05 * scale).float()


def _const_actor(c):
    import torch
    v = torch.zeros(A_N)
    v[-2:] = torch.atanh(torch.tensor(c, dtype=torch.float32))
    return v


def _ptr(t):
    return None if t is None else t.data_ptr()


# ---------------------------------------------------------------- CPU ------------------------------------------------------------------
def _args(**kw):
    from skillshot_learning_b200 import _lib
    Q = 4096
    a = _lib.PoolRolloutArgs()
    a.state, a.n_envs, a.pool_envs, a.n_opponents, a.params, a.opp_params, a.opp_param_stride = Q, 96, 48, 3, Q, Q, STRIDE
    a.obs, a.act, a.reward, a.opp_obs, a.opp_act, a.done, a.winner = Q, Q, Q, Q, Q, Q, Q
    a.n_ticks, a.noise_group, a.tensor_cores, a.reward_mode, a.tick_limit = 4, 128, 1, 1, 100
    for k, v in kw.items():
        setattr(a, k, v)
    return a


def test_pool_entry_points_reject_bad_arguments_without_a_gpu():
    from skillshot_learning_b200 import _lib
    L = _lib.lib
    P = 4096

    def step(n=96, M=48, K=3, act=P, opp=P, obs=P, obs2=None, rew=P, oobs=P, mode=1, reset=1, status=None, flags=0, stats=None):
        return L.ss_env_step_pool(P, n, M, K, act, opp, obs, obs2, rew, None, oobs, None, None, mode, 100, reset, 0, 0, status, flags,
                                  stats, None)
    bad = [dict(n=0), dict(M=-6), dict(M=102, n=96), dict(M=45), dict(K=0), dict(K=65, M=130, n=200), dict(act=None), dict(obs=None),
           dict(opp=None), dict(oobs=None), dict(mode=3), dict(mode=4), dict(reset=2), dict(obs=P + 8), dict(obs2=P + 4),
           dict(oobs=P + 8), dict(act=P + 4), dict(opp=P + 4), dict(rew=P + 2), dict(stats=P + 4), dict(status=P + 2),
           dict(status=P + 4, flags=2)]
    for kw in bad:
        assert step(**kw) == -1, kw
    assert L.ss_pool_rollout(None, None) == -1
    bad = [dict(state=None), dict(params=None), dict(obs=None), dict(act=None), dict(reward=None), dict(done=None), dict(winner=None),
           dict(opp_params=None), dict(opp_obs=None), dict(opp_act=None), dict(n_envs=0), dict(n_ticks=0), dict(pool_envs=45),
           dict(pool_envs=-6), dict(pool_envs=102), dict(n_opponents=0), dict(n_opponents=65, pool_envs=130, n_envs=200),
           dict(opp_param_stride=STRIDE + 2), dict(opp_param_stride=1024), dict(speeds=P), dict(reward_mode=3), dict(reset_mode=2),
           dict(param_noise_sd=0.5, noise_group=100), dict(param_noise_sd=0.5, noise_group=0), dict(param_noise_sd=-1.0),
           dict(state=P + 8), dict(obs=P + 4), dict(opp_obs=P + 8), dict(params=P + 4), dict(act=P + 4), dict(reward=P + 2),
           dict(pool_stats=P + 4), dict(status=P + 4, step_flags=2),
           # the ring: capacity and write position multiples of L = 2 S + M = 144, two segments unless one tick
           dict(ring_obs=P, ring_act=P, ring_reward=P, ring_next_obs=P, ring_done=P, capacity=144 * 3 + 2),
           dict(ring_obs=P, ring_act=P, ring_reward=P, ring_next_obs=P, ring_done=P, capacity=144 * 3, write_pos=10),
           dict(ring_obs=P, ring_act=P, ring_reward=P, ring_next_obs=P, ring_done=P, capacity=144 * 3, write_pos=144 * 3),
           dict(ring_obs=P, ring_act=P, ring_reward=P, ring_next_obs=P, ring_done=P, capacity=144),
           dict(ring_obs=P, ring_act=None, ring_reward=P, ring_next_obs=P, ring_done=P, capacity=288)]
    for kw in bad:
        a = _args(**kw)
        assert L.ss_pool_rollout(ctypes.byref(a), None) == -1, kw


def test_pool_argument_block_matches_the_header():
    """The ctypes mirror of struct ss_pool_rollout_args lists the header's fields in the header's order."""
    from skillshot_learning_b200 import _lib
    text = open(os.path.join(ROOT, "include", "skillshot_b200.h")).read()
    body = re.search(r"typedef struct ss_pool_rollout_args \{(.*?)\} ss_pool_rollout_args;", text, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = []
    for decl in body.split(";"):
        decl = decl.strip()
        if decl:
            names += [re.sub(r"[\s\*]|const", "", part.split()[-1]) for part in decl.split(",")]
    assert names == [f[0] for f in _lib.PoolRolloutArgs._fields_]
    assert _lib.POOL_STATS == int(re.search(r"#define SS_POOL_STATS (\d+)", text).group(1))


@pytest.mark.parametrize("n,M,K", [(10, 0, 3), (64, 32, 1), (100, 48, 3), (4096, 4096, 16), (130, 128, 64)])
def test_pool_layout_is_a_seat_balanced_permutation(n, M, K):
    from skillshot_learning_b200.learner import pool_layout
    rows = pool_layout(n, M, K)
    S, L, b = n - M, 2 * n - M, (M // K if M else 0)
    assert sorted(rows.reshape(-1).tolist()) == list(range(2 * n))
    assert np.array_equal(rows[:S], np.arange(2 * S).reshape(S, 2))
    for k in range(K if M else 0):
        blk = rows[S + k * b:S + (k + 1) * b]
        learner = blk < L
        assert (learner.sum(1) == 1).all()                                  # one learner and one opponent player per env
        assert learner[:b // 2, 0].all() and learner[b // 2:, 1].all()      # seat-balanced: player 1 first, then player 2
        assert np.array_equal(np.sort(blk[~learner]), L + np.arange(k * b, (k + 1) * b))     # one contiguous opponent segment
    assert np.array_equal(np.sort(rows[S:][rows[S:] < L]), np.arange(2 * S, L))


def test_trainer_rejects_what_the_pool_does_not_support_without_a_gpu():
    from skillshot_learning_b200 import SelfPlayTrainer
    a = _actor(1)
    for kw in (dict(frames=2), dict(process_group=object()), dict(reward_mode="simple"), dict(pool_envs=32), dict(pool_envs=130),
               dict(replay_capacity=1000), dict(replay_capacity=96)):
        with pytest.raises(ValueError):
            SelfPlayTrainer(64, device="cpu", opponents=[a, a, a], **kw)
    with pytest.raises(ValueError):
        SelfPlayTrainer(64, device="cpu", opponents=[a] * 65)
    with pytest.raises(ValueError):
        SelfPlayTrainer(64, device="cpu", opponents=[a, np.zeros(int(36482 + 12 * 256))])     # a 2-frame opponent


# ---------------------------------------------------------------- GPU helpers ----------------------------------------------------------
class _Both:
    """The same envs stepped by ss_env_step_ring ([n][2] rows) and by ss_env_step_pool (the pool layout)."""

    def __init__(self, n, M, K, mode="looking", random_positions=True, tick_limit=40, seed=3):
        import torch
        from skillshot_learning_b200 import SkillshotEnvs
        from skillshot_learning_b200.learner import pool_layout
        self.n, self.M, self.K, self.L = n, M, K, 2 * n - M
        self.mode, self.limit, self.seed, self.reset = MODES[mode], tick_limit, seed, 1 if random_positions else 0
        self.env = SkillshotEnvs(n, random_positions=random_positions, seed=seed)
        self.state_ring = self.env.state.clone()
        self.state_pool = self.env.state.clone()
        self.rows = torch.from_numpy(pool_layout(n, M, K).reshape(-1)).cuda()
        d = dict(device="cuda")
        self.ring = dict(obs=torch.zeros(2 * n, 12, **d), obs2=torch.zeros(2 * n, 12, **d), reward=torch.zeros(2 * n, **d),
                         done=torch.zeros(n, dtype=torch.uint8, **d), done_rows=torch.zeros(2 * n, dtype=torch.uint8, **d),
                         winner=torch.zeros(n, dtype=torch.uint8, **d), status=torch.zeros(2 + 144, dtype=torch.int32, **d))
        self.pool = dict(obs=torch.zeros(self.L, 12, **d), obs2=torch.zeros(self.L, 12, **d), reward=torch.zeros(self.L, **d),
                         done=torch.zeros(n, dtype=torch.uint8, **d), done_rows=torch.zeros(self.L, dtype=torch.uint8, **d),
                         winner=torch.zeros(n, dtype=torch.uint8, **d), status=torch.zeros(2 + 144, dtype=torch.int32, **d),
                         opp_obs=torch.zeros(max(M, 1), 12, **d), stats=torch.zeros(max(K, 1), 8, dtype=torch.int64, **d))
        self.counter = 100

    def tick(self, act):
        """act float32 [n, 2, 2] on the device; returns nothing, checks equality."""
        import torch
        from skillshot_learning_b200._lib import lib
        R, Q = self.ring, self.pool
        assert lib.ss_env_step_ring(self.state_ring.data_ptr(), self.n, act.data_ptr(), R["obs"].data_ptr(), R["obs2"].data_ptr(),
                                    R["reward"].data_ptr(), R["done"].data_ptr(), R["done_rows"].data_ptr(), R["winner"].data_ptr(), 1,
                                    self.mode, self.limit, 1, self.reset, self.seed, self.counter, None, R["status"].data_ptr(), 2,
                                    None) == 0
        comb = torch.empty(2 * self.n, 2, device="cuda")
        comb[self.rows] = act.reshape(-1, 2)
        la, oa = comb[:self.L].contiguous(), comb[self.L:].contiguous()
        assert lib.ss_env_step_pool(self.state_pool.data_ptr(), self.n, self.M, self.K, la.data_ptr(), _ptr(oa) if self.M else None,
                                    Q["obs"].data_ptr(), Q["obs2"].data_ptr(), Q["reward"].data_ptr(), Q["done_rows"].data_ptr(),
                                    Q["opp_obs"].data_ptr(), Q["done"].data_ptr(), Q["winner"].data_ptr(), self.mode, self.limit,
                                    self.reset, self.seed, self.counter, Q["status"].data_ptr(), 2, Q["stats"].data_ptr(), None) == 0
        self.counter += 1
        torch.cuda.synchronize()
        assert torch.equal(self.state_ring, self.state_pool)
        assert torch.equal(R["done"], Q["done"]) and torch.equal(R["winner"], Q["winner"]) and torch.equal(R["status"], Q["status"])
        obs = torch.cat([Q["obs"], Q["opp_obs"][:self.M]])[self.rows]
        assert torch.equal(obs, R["obs"]) and torch.equal(Q["obs2"], Q["obs"])
        learner = self.rows < self.L
        lr = self.rows[learner]
        assert torch.equal(Q["done_rows"][lr], R["done_rows"][learner])
        if self.mode:
            assert torch.equal(Q["reward"][lr], R["reward"][learner])


def _crafted_double_hits(env, envs):
    """Puts the games of `envs` one tick before a double hit: each projectile 5 pixels below the other player, flying up,
    both cooldowns running.  With zero actions both players are hit on the next tick (winner_id 1: player 1 is recorded)."""
    st = env.export_state()
    for e in envs:
        st["px"][e], st["py"][e] = (60, 180), (60, 180)
        st["qx"][e], st["qy"][e] = (180, 60), (185, 65)
        st["qrot"][e] = (0.0, 0.0)
        st["valid"][e], st["cd"][e], st["live"][e], st["winner"][e], st["ticks"][e] = (1, 1), (10, 10), 1, 0, 7
    env.import_state(st)


# ---------------------------------------------------------------- GPU ------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["none", "looking", "terminal"])
@pytest.mark.parametrize("random_positions", [False, True])
def test_pool_step_without_pool_envs_is_the_ring_step(mode, random_positions):
    import torch
    b = _Both(1000, 0, 0, mode=mode, random_positions=random_positions)
    g = torch.Generator(device="cuda").manual_seed(1)
    for _ in range(60):
        b.tick(torch.rand(1000, 2, 2, device="cuda", generator=g) * 2.4 - 1.2)


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 3, 16])
def test_pool_step_is_the_ring_step_under_the_layout(K):
    import torch
    n, M = 3000 + 96 * K, 96 * K
    b = _Both(n, M, K, mode="looking", tick_limit=25)
    g = torch.Generator(device="cuda").manual_seed(K)
    for _ in range(70):                                  # several auto-resets at the tick limit
        b.tick(torch.rand(n, 2, 2, device="cuda", generator=g) * 2.4 - 1.2)


@pytest.mark.gpu
def test_pool_counters_equal_a_host_tally():
    import torch
    n, M, K = 1200, 960, 5
    S, b = n - M, M // K
    both = _Both(n, M, K, mode="terminal", random_positions=False, tick_limit=30)
    crafted = [S + k * b + q for k in range(K) for q in (0, 3, b - 1, b - 4)]        # learner as player 1 and as player 2
    env = both.env
    env.state.copy_(both.state_pool)
    _crafted_double_hits(env, crafted)
    both.state_ring.copy_(env.state)
    both.state_pool.copy_(env.state)
    length = env.export_state()["ticks"].astype(np.int64)
    tally = np.zeros((K, 8), np.int64)
    g = torch.Generator(device="cuda").manual_seed(7)
    doubles = 0
    for t in range(80):
        act = torch.rand(n, 2, 2, device="cuda", generator=g) * 2.4 - 1.2
        if t == 0:
            act[crafted] = 0.0
        both.tick(act)
        done, winner = both.pool["done"].cpu().numpy(), both.pool["winner"].cpu().numpy()
        length += 1
        for j in np.nonzero(done[S:])[0]:
            k, lp = j // b, int(j % b >= b // 2)
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
    assert np.array_equal(both.pool["stats"].cpu().numpy(), tally)


def _pool_setup(n, M, K, precision, capacity_segs, seed=5):
    import torch
    from skillshot_learning_b200 import SkillshotEnvs
    from skillshot_learning_b200.learner import pool_layout
    L = 2 * n - M
    env = SkillshotEnvs(n, random_positions=True, seed=seed)
    rows = torch.from_numpy(pool_layout(n, M, K).reshape(-1)).cuda()
    obs = torch.empty(2 * n, 12, device="cuda")
    obs[rows] = env.observe().reshape(-1, 12)
    opp = torch.zeros(max(K, 1), STRIDE, device="cuda")
    for k in range(K):
        opp[k, :A_N] = _actor(40 + k, scale=4.0).cuda()
    cap = capacity_segs * L
    d = dict(device="cuda")
    ring = dict(obs=torch.zeros(cap, 12, **d), act=torch.zeros(cap, 2, **d), reward=torch.zeros(cap, **d),
                next_obs=torch.zeros(cap, 12, **d), done=torch.zeros(cap, dtype=torch.uint8, **d))
    return dict(env=env, L=L, obs=obs, opp=opp, ring=ring, cap=cap, params=_actor(9, scale=3.0).cuda(),
                status=torch.zeros(2 + 144, dtype=torch.int32, **d), stats=torch.zeros(max(K, 1), 8, dtype=torch.int64, **d),
                act=torch.zeros(2 * n, 2, **d), reward=torch.zeros(L, **d), done=torch.zeros(n, dtype=torch.uint8, **d),
                winner=torch.zeros(n, dtype=torch.uint8, **d), n=n, M=M, K=K, tc=1 if precision == "bf16" else 0)


def _rollout_args(s, n_ticks, write_pos, env_counter, noise_counter):
    from skillshot_learning_b200 import _lib
    L, r = s["L"], s["ring"]
    a = _lib.PoolRolloutArgs()
    a.state, a.n_envs, a.pool_envs, a.n_opponents = s["env"].state.data_ptr(), s["n"], s["M"], s["K"]
    a.params, a.opp_params, a.opp_param_stride = s["params"].data_ptr(), s["opp"].data_ptr(), STRIDE
    a.obs, a.act, a.reward = s["obs"].data_ptr(), s["act"].data_ptr(), s["reward"].data_ptr()
    a.opp_obs, a.opp_act = s["obs"][L:].data_ptr(), s["act"][L:].data_ptr()
    a.done, a.winner = s["done"].data_ptr(), s["winner"].data_ptr()
    a.ring_obs, a.ring_act, a.ring_reward, a.ring_next_obs, a.ring_done = (r[k].data_ptr() for k in ("obs", "act", "reward", "next_obs", "done"))
    a.capacity, a.write_pos, a.n_ticks = s["cap"], write_pos, n_ticks
    a.param_noise_sd, a.noise_group, a.tensor_cores, a.reward_mode, a.tick_limit = 0.5, 128, s["tc"], 1, 60
    a.reset_mode, a.env_seed, a.env_counter, a.noise_seed, a.noise_counter = 1, 5, env_counter, 11, noise_counter
    a.status, a.step_flags, a.pool_stats = s["status"].data_ptr(), 2, s["stats"].data_ptr()
    return a


def _stepwise(s, n_ticks, write_pos, env_counter, noise_counter):
    """ss_pool_rollout composed from its three entry points, tick by tick."""
    import torch
    from skillshot_learning_b200._lib import lib
    n, M, K, L, r = s["n"], s["M"], s["K"], s["L"], s["ring"]
    segs = s["cap"] // L
    seg = write_pos // L
    r["obs"][seg * L:(seg + 1) * L] = s["obs"][:L]
    b = M // K if M else 0
    seg_rows = (ctypes.c_int64 * max(K, 1))(*([b] * max(K, 1)))
    for t in range(n_ticks):
        o, a = r["obs"][seg * L:(seg + 1) * L], r["act"][seg * L:(seg + 1) * L]
        nxt = (seg + 1) % segs
        o_next = r["obs"][nxt * L:(nxt + 1) * L] if t + 1 < n_ticks else s["obs"][:L]
        fwd = lib.ss_actor_forward_tc if s["tc"] else lib.ss_actor_forward
        assert fwd(s["params"].data_ptr(), o.data_ptr(), a.data_ptr(), L, 0.5, 128, 0.0, 11, noise_counter + t, None) == 0
        oo, oa = s["obs"][L:], s["act"][L:]
        if M:
            if s["tc"]:
                assert lib.ss_actor_forward_segments_tc(s["opp"].data_ptr(), STRIDE, seg_rows, K, oo.data_ptr(), oa.data_ptr(), None) == 0
            else:
                for k in range(K):
                    assert lib.ss_actor_forward(s["opp"][k].data_ptr(), oo[k * b:].data_ptr(), oa[k * b:].data_ptr(), b, 0.0, 1, 0.0, 0, 0,
                                                None) == 0
        assert lib.ss_env_step_pool(s["env"].state.data_ptr(), n, M, K, a.data_ptr(), oa.data_ptr() if M else None,
                                    r["next_obs"][seg * L:].data_ptr(), o_next.data_ptr(), r["reward"][seg * L:].data_ptr(),
                                    r["done"][seg * L:].data_ptr(), oo.data_ptr() if M else None, s["done"].data_ptr(),
                                    s["winner"].data_ptr(), 1, 60, 1, 5, env_counter + t, s["status"].data_ptr(), 2,
                                    s["stats"].data_ptr(), None) == 0
        seg = nxt
    last = (seg + segs - 1) % segs
    s["act"][:L] = r["act"][last * L:(last + 1) * L]
    s["reward"].copy_(r["reward"][last * L:(last + 1) * L])
    torch.cuda.synchronize()


def _same(s1, s2):
    import torch
    for k in ("obs", "act", "reward", "done", "winner", "status", "stats"):
        assert torch.equal(s1[k], s2[k]), k
    assert torch.equal(s1["env"].state, s2["env"].state)
    for k in s1["ring"]:
        assert torch.equal(s1["ring"][k], s2["ring"][k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["bf16", "f32"])
@pytest.mark.parametrize("n_ticks", [5, 6])
def test_pool_rollout_equals_its_stepwise_composition(precision, n_ticks):
    from skillshot_learning_b200._lib import lib
    n, M, K = 2560, 1536, 6
    one, two = _pool_setup(n, M, K, precision, 3), _pool_setup(n, M, K, precision, 3)
    L = one["L"]
    pos, ec, nc = L, 7, 13
    for rep in range(2):                                  # the ring wraps (3 segments, 2 x n_ticks ticks from segment 1)
        a = _rollout_args(one, n_ticks, pos, ec, nc)
        assert lib.ss_pool_rollout(ctypes.byref(a), None) == 0
        _stepwise(two, n_ticks, pos, ec, nc)
        _same(one, two)
        pos, ec, nc = (pos + n_ticks * L) % one["cap"], ec + n_ticks, nc + n_ticks
    assert one["stats"][:, 0].sum() > 0


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["bf16", "f32"])
def test_pool_rollout_without_pool_envs_is_the_selfplay_rollout(precision):
    import torch
    from skillshot_learning_b200._lib import lib
    n, T = 3000, 50
    s = _pool_setup(n, 0, 0, precision, 4)
    ref = _pool_setup(n, 0, 0, precision, 4)
    a = _rollout_args(s, T, 2 * (2 * n), 3, 4)
    assert lib.ss_pool_rollout(ctypes.byref(a), None) == 0
    r = ref["ring"]
    obs_b = torch.empty_like(ref["obs"])
    assert lib.ss_selfplay_rollout(ref["env"].state.data_ptr(), n, ref["params"].data_ptr(), ref["obs"].data_ptr(), obs_b.data_ptr(),
                                   ref["act"].data_ptr(), ref["reward"].data_ptr(), ref["done"].data_ptr(), ref["winner"].data_ptr(),
                                   r["obs"].data_ptr(), r["act"].data_ptr(), r["reward"].data_ptr(), r["next_obs"].data_ptr(),
                                   r["done"].data_ptr(), ref["cap"], 2 * (2 * n), T, 0.5, 128, 0.0, ref["tc"], 1, 60, 1, 5, 3, 11, 4,
                                   None, ref["status"].data_ptr(), 2, None) == 0
    torch.cuda.synchronize()
    _same(s, ref)
    assert int(s["status"][2:].view(torch.int64)[0]) > 0                    # episodes ended


@pytest.mark.gpu
def test_constant_action_opponents_equal_the_oracle():
    """The learner's actions read back from the ring and the opponents' constant actions replayed through the C oracle
    give the same positions, winners, rewards and hit flags."""
    import torch
    from oracle.oracle import OracleEnvs
    from skillshot_learning_b200._lib import lib
    from skillshot_learning_b200.learner import pool_layout
    n, M, K, T = 800, 512, 2, 40
    S = n - M
    consts = [(0.898, -0.08), (0.189, -0.324)]
    s = _pool_setup(n, M, K, "bf16", T + 1)
    L = s["L"]
    s["env"].reset(random_positions=False)
    rows = torch.from_numpy(pool_layout(n, M, K).reshape(-1)).cuda()
    s["obs"][rows] = s["env"].observe().reshape(-1, 12)
    for k, c in enumerate(consts):
        s["opp"][k, :A_N] = _const_actor(c).cuda()
    a = _rollout_args(s, T, 0, 0, 0)
    a.reward_mode, a.reset_mode, a.tick_limit = 2, 0, 25
    assert lib.ss_pool_rollout(ctypes.byref(a), None) == 0
    opp_act = s["act"][L:].cpu().numpy()
    assert all((opp_act[k * (M // K):(k + 1) * (M // K)] == opp_act[k * (M // K)]).all() for k in range(K))
    ring = {k: v.cpu().numpy() for k, v in s["ring"].items()}
    lay = pool_layout(n, M, K)
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
    want, got = orc.snapshot(), s["env"].export_state()
    for k in ("px", "py", "qx", "qy", "ticks", "live", "winner"):
        assert np.array_equal(got[k], want[k]), k
    assert s["stats"][:, 0].sum() > 0 and S > 0


def _trainer(**kw):
    from skillshot_learning_b200 import SelfPlayTrainer
    args = dict(seed=3, batch_size=1024, precision="bf16", tick_limit=120, opponents=[_actor(20 + k, scale=4.0) for k in range(3)])
    args.update(kw)
    return SelfPlayTrainer(2048, **args)


def _same_trainer(t1, t2):
    import torch
    assert torch.equal(t1.networks.params, t2.networks.params) and torch.equal(t1.networks.target, t2.networks.target)
    assert torch.equal(t1.envs.state, t2.envs.state) and torch.equal(t1.replay.obs, t2.replay.obs)
    assert torch.equal(t1.replay.next_obs, t2.replay.next_obs) and torch.equal(t1.replay.reward, t2.replay.reward)
    assert torch.equal(t1.obs, t2.obs) and torch.equal(t1.pool_stats, t2.pool_stats) and torch.equal(t1.opponents, t2.opponents)
    assert t1.envs.counter == t2.envs.counter and t1.networks.counter == t2.networks.counter
    assert t1.replay.pos == t2.replay.pos and t1.replay.size == t2.replay.size


@pytest.mark.gpu
def test_trainer_checkpoint_with_a_pool_resumes_bit_identically():
    import torch
    t1 = _trainer()
    assert t1.pool_envs == 1020 and t1.replay.capacity == 8 * (2 * 2048 - 1020)
    for _ in range(3):
        t1.rollout(3)
        t1.update()
    torch.cuda.synchronize()
    sd = t1.state_dict()
    for _ in range(3):
        t1.rollout(3)
        t1.update()
    t2 = _trainer(seed=8, opponents=[_actor(50 + k) for k in range(3)])
    t2.load_state_dict(sd)
    for _ in range(3):
        t2.rollout(3)
        t2.update()
    torch.cuda.synchronize()
    _same_trainer(t1, t2)
    prog = t1.pool_progress()
    assert len(prog) == 3 and sum(p["episodes"] for p in prog) > 0
    assert all(p["episodes"] == p["wins"] + p["losses"] + p["draws"] for p in prog)
    with pytest.raises(ValueError):
        _trainer(opponents=[_actor(1)] * 2).load_state_dict(sd)            # another pool layout
    with pytest.raises(ValueError):
        _trainer(opponents=None).load_state_dict(sd)


@pytest.mark.gpu
def test_set_opponent_takes_effect_on_the_next_tick():
    import torch
    new = _actor(77, scale=4.0)
    t1, t2, t3 = _trainer(), _trainer(), _trainer()
    t1.rollout(4)
    t1.set_opponent(1, new)
    t1.rollout(5)
    for _ in range(4):
        t2.rollout_tick()
    t2.set_opponent(1, [w.numpy() for w in _split(new)])
    for _ in range(5):
        t2.rollout_tick()
    t3.rollout(9)
    torch.cuda.synchronize()
    _same_trainer(t1, t2)
    assert not torch.equal(t1.envs.state, t3.envs.state)


def _split(v):
    shapes = [(12, 256), (256,), (256, 128), (128,), (128, 2), (2,)]
    out, o = [], 0
    for sh in shapes:
        k = int(np.prod(sh))
        out.append(v[o:o + k].reshape(sh))
        o += k
    return out


@pytest.mark.gpu
def test_evaluate_league_does_not_disturb_pool_training():
    import torch

    def run(evaluate):
        tr = _trainer()
        for k in range(4):
            tr.rollout(4)
            tr.update()
            if evaluate and k == 1:
                tr.evaluate_league([_actor(90 + s) for s in range(2)], games_per_pair=512, seed=2, tick_limit=100)
        torch.cuda.synchronize()
        return tr
    _same_trainer(run(True), run(False))
