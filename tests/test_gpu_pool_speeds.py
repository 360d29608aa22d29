"""Training against a pool with per-env game speeds (ss_env_step_pool_speeds, ss_pool_rollout_speeds and
SelfPlayTrainer with envs.set_speeds).  The GPU tests compare with ==: the speeds step with the reference constants against
ss_env_step_pool_blocks, with a random speed sweep against ss_env_step_ring under the layout's permutation, its counters
against a host tally, constant-action opponents against the C oracle, ss_pool_restart against an auto-reset tick and
ss_env_reset, the one-call rollout against its stepwise composition, and the trainer's one-call rollout and checkpoints
against per-tick and uninterrupted runs.  The unmarked tests run without a GPU: argument rejection and the trainer's
refusals."""
import ctypes

import numpy as np
import pytest

from tests.test_gpu_pool import MODES, _crafted_double_hits
from tests.test_gpu_pool_blocks import _BlockSetup, _blocks, _export, _table
from tests.test_gpu_pool_frames import _actor, _const_actor, _n_params, _same, _same_pool

REFERENCE = (3.0, 0.25, 5.0, 15)


def _sweep(n, seed):
    """config-5 style per-env speeds: each constant U(0.5, 2) times the reference's, the cooldown rounded, at least 1"""
    rng = np.random.default_rng(seed)
    s = lambda: rng.uniform(0.5, 2.0, n)
    return 3.0 * s(), 0.25 * s(), 5.0 * s(), np.maximum(np.round(15.0 * s()), 1).astype(np.int64)


# ---------------------------------------------------------------- CPU ------------------------------------------------------------------
def _args(**kw):
    """a valid argument block (n 96, M 48, K 3 -> L 144, b 16) of fake device pointers, a 4-frame learner, opponent frames
    {1, 20, 1}, tensor cores, parameter noise in groups of 128, per-env speeds"""
    from skillshot_learning_b200 import _lib
    Q = 4096
    a = _lib.PoolRolloutFramesArgs()
    a.state, a.n_envs, a.pool_envs, a.n_opponents, a.params, a.opp_params, a.opp_param_stride = Q, 96, 48, 3, Q, Q, 94852
    a.obs, a.act, a.reward, a.opp_obs, a.opp_act, a.done, a.winner = Q, Q, Q, Q, Q, Q, Q
    a.n_ticks, a.noise_group, a.param_noise_sd, a.tensor_cores, a.reward_mode, a.tick_limit = 4, 128, 0.5, 1, 1, 100
    a.frames, a.stack_tc, a.stack32, a.rows, a.head, a.speeds = 4, Q, Q, Q, 0, Q
    frames = kw.pop("opp_frames", [1, 20, 1])
    stacks = kw.pop("opp_stacks", [None if f == 1 else Q for f in frames])
    a._keep = ((ctypes.c_int * len(frames))(*frames), (ctypes.c_void_p * len(stacks))(*stacks))
    a.opp_frames, a.opp_stacks = a._keep
    for k, v in kw.items():
        setattr(a, k, v)
    if "workspace" not in kw:
        a.workspace, a.workspace_bytes = Q, 1 << 40
    return a


def test_pool_speeds_entry_points_reject_bad_arguments_without_a_gpu():
    from skillshot_learning_b200 import _lib
    L, P = _lib.lib, 4096

    def step(speeds=P, mode=1, table=None, M=48, K=3, n=96):
        return L.ss_env_step_pool_speeds(P, n, M, K, P, P, P, None, P, None, P, None, None, mode, 100, 1, 0, 0, None, 0, None, table,
                                         speeds, None)
    bad_tables = ([16, 15, 17], [16, 16, 18], [16, 16, 14])
    for kw in (dict(speeds=None), dict(speeds=P + 8), dict(mode=3), dict(mode=4), dict(mode=-1), dict(M=50), dict(M=97),
               dict(K=65, M=130, n=200), dict(K=0)):
        assert step(**kw) == -1, kw
    for blocks in bad_tables:
        assert step(table=_table(blocks)) == -1, blocks
    assert step(table=_table([2] * 65), M=130, K=65, n=200) == -1
    assert step(table=_table([16, 16, 16]), M=0) == -1                  # no pool envs take no table
    assert L.ss_pool_rollout_speeds(None, None) == -1
    ring = dict(ring_obs=P, ring_act=P, ring_reward=P, ring_next_obs=P, ring_done=P)
    need = L.ss_pool_rollout_frames_workspace_bytes(ctypes.byref(_args()))
    assert need == L.ss_pool_rollout_frames_workspace_bytes(ctypes.byref(_args(speeds=None)))
    # the rules of ss_pool_rollout_frames, then the speeds' own
    bad = [dict(frames=0), dict(frames=21), dict(opp_frames=[1, 0, 1]), dict(opp_frames=[1, 21, 1]),
           dict(stack_tc=None), dict(stack32=None), dict(rows=None), dict(opp_stacks=[None, None, None]),
           dict(stack32=P + 4), dict(opp_stacks=[None, P + 8, None]), dict(head=-1), dict(action_noise_sd=0.1),
           dict(workspace=None), dict(workspace=P, workspace_bytes=need - 16), dict(workspace=P + 8, workspace_bytes=need),
           dict(opp_param_stride=36484), dict(noise_group=100), dict(noise_group=0), dict(reward_mode=3),
           dict(n_opponents=65, pool_envs=130, n_envs=200, opp_frames=[1] * 65), dict(pool_envs=45), dict(pool_envs=50),
           dict(capacity=144 * 3 + 2, **ring), dict(capacity=144 * 3, write_pos=10, **ring), dict(capacity=144, **ring),
           dict(speeds=None), dict(speeds=P + 8)]
    bad += [dict(opp_envs=_table(b)) for b in bad_tables]
    for kw in bad:
        assert L.ss_pool_rollout_speeds(ctypes.byref(_args(**kw)), None) == -1, kw
    # ss_pool_rollout_frames still takes no speeds
    assert L.ss_pool_rollout_frames(ctypes.byref(_args()), None) == -1


def test_pool_trainer_refusals_hold_without_a_gpu():
    from skillshot_learning_b200 import SelfPlayTrainer
    opp = [_actor(1), _actor(2, frames=20)]
    for kw in (dict(process_group=object()), dict(reward_mode="simple")):
        with pytest.raises(ValueError):
            SelfPlayTrainer(64, frames=20, opponents=opp, **kw)


# ---------------------------------------------------------------- GPU: the step ---------------------------------------------------------
class _Steps:
    """The same envs with the same per-env speeds stepped by ss_env_step_ring ([n][2] rows) and by ss_env_step_pool_speeds
    under `blocks` (None: the NULL table, M / K each); with reference=True also by ss_env_step_pool_blocks without speeds."""

    def __init__(self, n, M, K, blocks=None, mode="looking", random_positions=True, tick_limit=40, flags=2, speeds=None, seed=3,
                 reference=False):
        import torch
        from skillshot_learning_b200 import SkillshotEnvs
        from skillshot_learning_b200.learner import pool_layout
        self.n, self.M, self.K, self.L, self.S = n, M, K, 2 * n - M, n - M
        self.blocks = blocks if blocks is not None else ([M // K] * K if M else [])
        self.mode, self.limit, self.seed, self.reset, self.flags = MODES[mode], tick_limit, seed, 1 if random_positions else 0, flags
        self.reference = reference
        self.env = SkillshotEnvs(n, random_positions=random_positions, seed=seed)
        self.env.set_speeds(*(speeds if speeds is not None else _sweep(n, seed)))
        self.speeds = self.env.speeds
        self.states = dict(ring=self.env.state.clone(), speeds=self.env.state.clone(), blocks=self.env.state.clone())
        self.rows = torch.from_numpy(pool_layout(n, M, K, blocks).reshape(-1)).cuda()
        d = dict(device="cuda")
        self.out = dict(ring=dict(obs=torch.zeros(2 * n, 12, **d), obs2=torch.zeros(2 * n, 12, **d), reward=torch.zeros(2 * n, **d),
                                  done=torch.zeros(n, dtype=torch.uint8, **d), done_rows=torch.zeros(2 * n, dtype=torch.uint8, **d),
                                  winner=torch.zeros(n, dtype=torch.uint8, **d), status=torch.zeros(2 + 144, dtype=torch.int32, **d)))
        for k in ("speeds", "blocks"):
            self.out[k] = dict(obs=torch.full((self.L, 12), -3.0, **d), obs2=torch.zeros(self.L, 12, **d),
                               reward=torch.full((self.L,), -5.0, **d), done=torch.zeros(n, dtype=torch.uint8, **d),
                               done_rows=torch.zeros(self.L, dtype=torch.uint8, **d), winner=torch.zeros(n, dtype=torch.uint8, **d),
                               status=torch.zeros(2 + 144, dtype=torch.int32, **d), opp_obs=torch.zeros(max(M, 1), 12, **d),
                               stats=torch.zeros(max(K, 1), 8, dtype=torch.int64, **d))
        self.table = None if blocks is None else _table(blocks)
        self.counter = 100

    def tick(self, act):
        import torch
        from skillshot_learning_b200._lib import lib
        R = self.out["ring"]
        assert lib.ss_env_step_ring(self.states["ring"].data_ptr(), self.n, act.data_ptr(), R["obs"].data_ptr(), R["obs2"].data_ptr(),
                                    R["reward"].data_ptr(), R["done"].data_ptr(), R["done_rows"].data_ptr(), R["winner"].data_ptr(), 1,
                                    self.mode, self.limit, 1, self.reset, self.seed, self.counter, self.speeds.data_ptr(),
                                    R["status"].data_ptr(), self.flags, None) == 0
        comb = torch.empty(2 * self.n, 2, device="cuda")
        comb[self.rows] = act.reshape(-1, 2)
        la, oa = comb[:self.L].contiguous(), comb[self.L:].contiguous()
        for k in ("speeds", "blocks") if self.reference else ("speeds",):
            Q = self.out[k]
            args = [self.states[k].data_ptr(), self.n, self.M, self.K, la.data_ptr(), oa.data_ptr() if self.M else None,
                    Q["obs"].data_ptr(), Q["obs2"].data_ptr(), Q["reward"].data_ptr(), Q["done_rows"].data_ptr(),
                    Q["opp_obs"].data_ptr() if self.M else None, Q["done"].data_ptr(), Q["winner"].data_ptr(), self.mode, self.limit,
                    self.reset, self.seed, self.counter, Q["status"].data_ptr(), self.flags, Q["stats"].data_ptr(), self.table]
            if k == "speeds":
                assert lib.ss_env_step_pool_speeds(*(args + [self.speeds.data_ptr(), None])) == 0
            else:
                assert lib.ss_env_step_pool_blocks(*(args + [None])) == 0
        self.counter += 1
        torch.cuda.synchronize()
        Q = self.out["speeds"]
        assert torch.equal(self.states["ring"], self.states["speeds"])
        assert torch.equal(R["done"], Q["done"]) and torch.equal(R["winner"], Q["winner"]) and torch.equal(R["status"], Q["status"])
        obs = torch.cat([Q["obs"], Q["opp_obs"][:self.M]])[self.rows]
        assert torch.equal(obs, R["obs"]) and torch.equal(Q["obs2"], Q["obs"])
        learner = self.rows < self.L
        lr = self.rows[learner]
        assert torch.equal(Q["done_rows"][lr], R["done_rows"][learner])
        if self.mode:
            assert torch.equal(Q["reward"][lr], R["reward"][learner])
        else:
            assert (Q["reward"] == -5.0).all()                              # reward none: not written
        if self.reference:
            assert torch.equal(self.states["blocks"], self.states["speeds"])
            for k, v in self.out["blocks"].items():
                assert torch.equal(v, Q[k]), k


def _ticks(s, T, seed):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    for _ in range(T):
        s.tick(torch.rand(s.n, 2, 2, device="cuda", generator=g) * 2.4 - 1.2)


@pytest.mark.gpu
@pytest.mark.parametrize("table", ["null", "skewed"])
@pytest.mark.parametrize("mode", ["none", "looking", "terminal"])
@pytest.mark.parametrize("K", [1, 3, 16, 64])
def test_reference_speeds_are_the_per_player_step(K, mode, table):
    """A speeds buffer of (3, 0.25, 5, 15) everywhere gives the bytes of ss_env_step_pool_blocks without speeds."""
    blocks = _blocks(K, K) if table == "skewed" else None
    M = sum(blocks) if blocks else 32 * K
    n = 1500 + M
    s = _Steps(n, M, K, blocks, mode=mode, random_positions=K % 2 == 1, tick_limit=25, flags=2 if K < 10 else 0,
               speeds=tuple(np.full(n, v) for v in REFERENCE), reference=True)
    _ticks(s, 60, K)                                     # several auto-resets at the tick limit
    assert s.out["speeds"]["stats"][:, 0].sum() > 0


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["none", "looking", "terminal"])
@pytest.mark.parametrize("K,table", [(1, "null"), (3, "skewed"), (16, "skewed"), (64, "null")])
def test_speed_sweep_is_the_ring_step_under_the_layout(K, table, mode):
    blocks = _blocks(K, K + 1) if table == "skewed" else None
    M = sum(blocks) if blocks else 32 * K
    n = 1500 + M
    s = _Steps(n, M, K, blocks, mode=mode, random_positions=K != 16, tick_limit=30, flags=2 if K < 10 else 0, seed=K)
    _ticks(s, 90, K)
    assert s.out["speeds"]["stats"][:, 0].sum() > 0


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["none", "looking", "terminal"])
def test_speeds_step_without_pool_envs_is_the_ring_step(mode):
    s = _Steps(1000, 0, 1, None, mode=mode, tick_limit=20)
    _ticks(s, 60, 2)
    assert (s.out["speeds"]["stats"] == 0).all()


@pytest.mark.gpu
def test_speeds_counters_equal_a_host_tally():
    import torch
    blocks = [8, 200, 12, 340, 400]
    n, M, K = 1200, sum(blocks), len(blocks)
    S = n - M
    starts = np.concatenate([[0], np.cumsum(blocks)])
    crafted = [S + int(starts[k]) + q for k in range(K) for q in (0, 3, blocks[k] - 1, blocks[k] - 4)]   # the learner in both seats
    sp = _sweep(n, 11)
    for a, v in zip(sp, REFERENCE):                       # the crafted games are set up for the reference speeds
        a[crafted] = v
    s = _Steps(n, M, K, blocks, mode="terminal", random_positions=False, tick_limit=30, speeds=sp)
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
        done, winner = s.out["speeds"]["done"].cpu().numpy(), s.out["speeds"]["winner"].cpu().numpy()
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
                assert w == 1                                     # a double hit records player 1 as hit
        length[done != 0] = 0
    assert doubles == len(crafted)
    assert tally[:, 1].sum() > 0 and tally[:, 2].sum() > 0 and tally[:, 3].sum() > 0
    assert np.array_equal(s.out["speeds"]["stats"].cpu().numpy(), tally)


@pytest.mark.gpu
@pytest.mark.parametrize("random_positions", [False, True])
def test_restart_with_speeds_is_an_auto_reset_and_an_env_reset(random_positions):
    """With per-env speeds, ss_pool_restart with counter c gives the state and observations of an ss_env_step_pool_speeds
    tick with counter c that ends (and so auto-resets) every game, and the state of ss_env_reset over the pool envs."""
    import torch
    from skillshot_learning_b200._lib import lib
    blocks = [6, 40, 2, 18, 30]
    n, M, K = 700, sum(blocks), len(blocks)
    S, L = n - M, 2 * n - M
    s = _Steps(n, M, K, blocks, mode="looking", random_positions=random_positions, tick_limit=1, seed=6)
    _ticks(s, 3, 4)                                      # (games of any state: every tick ends and restarts all of them)
    start = s.states["speeds"].clone()
    obs, opp = torch.full((L, 12), -7.0, device="cuda"), torch.full((M, 12), -7.0, device="cuda")
    obs0 = obs.clone()
    c, reset = s.counter, 1 if random_positions else 0
    assert lib.ss_pool_restart(start.data_ptr(), n, M, K, s.table, reset, s.seed, c, obs.data_ptr(), opp.data_ptr(), None, None) == 0
    _ticks(s, 1, 5)                                      # every game ends under counter c
    torch.cuda.synchronize()
    mine, tick = _export(s.env, start), _export(s.env, s.states["speeds"])
    for k in mine:
        assert np.array_equal(mine[k][S:], tick[k][S:]), k
    Q = s.out["speeds"]
    assert torch.equal(obs[2 * S:], Q["obs"][2 * S:]) and torch.equal(opp, Q["opp_obs"])
    assert torch.equal(obs[:2 * S], obs0[:2 * S])
    # the restarted games' cooldown observation is 0 whatever the env's cooldown_max
    assert (opp[:, 5] == 0).all() and (obs[2 * S:, 5] == 0).all()
    before = s.states["ring"].clone()
    ref = before.clone()
    mask = torch.zeros(n, dtype=torch.uint8, device="cuda")
    mask[S:] = 1
    assert lib.ss_env_reset(ref.data_ptr(), n, mask.data_ptr(), reset, None, s.seed, c + 1, None) == 0
    again = before.clone()
    assert lib.ss_pool_restart(again.data_ptr(), n, M, K, s.table, reset, s.seed, c + 1, obs.data_ptr(), opp.data_ptr(), None, None) == 0
    torch.cuda.synchronize()
    assert torch.equal(again, ref)


@pytest.mark.gpu
def test_constant_action_opponents_with_a_speed_sweep_equal_the_oracle():
    import torch
    from oracle.oracle import OracleEnvs
    from skillshot_learning_b200._lib import lib
    from skillshot_learning_b200.learner import pool_layout
    n, T = 800, 40
    blocks = [64, 300, 148]
    consts = [((0.898, -0.08), 20), ((0.189, -0.324), 1), ((-0.5, 0.7), 4)]
    sp = _sweep(n, 21)
    s = _SpeedSetup(n, blocks, 4, [f for _, f in consts], "bf16", T + 1, speeds=sp)
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
    assert lib.ss_pool_rollout_speeds(ctypes.byref(a), None) == 0
    torch.cuda.synchronize()
    opp_act = s.act[L:].cpu().numpy()
    assert all((opp_act[s.starts[k]:s.starts[k + 1]] == opp_act[s.starts[k]]).all() for k in range(K))
    ring = {k: v.cpu().numpy() for k, v in s.ring.items()}
    learner = lay < L
    orc = OracleEnvs(n)
    orc.set_speeds(*sp)
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
    for k in ("px", "py", "qx", "qy", "cd", "ticks", "live", "winner"):
        assert np.array_equal(got[k], want[k]), k
    assert s.stats[:, 0].sum() > 0 and S > 0


# ---------------------------------------------------------------- GPU: the rollout -----------------------------------------------------
class _SpeedSetup(_BlockSetup):
    """_BlockSetup with per-env speeds: the one-call rollout is ss_pool_rollout_speeds, and the stepwise composition steps
    the envs with ss_env_step_pool_speeds where _BlockSetup's calls ss_env_step_pool_blocks."""

    def __init__(self, n, blocks, frames, opp_frames, precision, segs, table=True, speeds=None, seed=5):
        super().__init__(n, blocks, frames, opp_frames, precision, segs, table, seed)
        self.env.set_speeds(*(speeds if speeds is not None else _sweep(n, seed)))

    def args(self, n_ticks, write_pos, env_counter, noise_counter):
        a = super().args(n_ticks, write_pos, env_counter, noise_counter)
        a.speeds = self.env.speeds.data_ptr()
        return a

    def run(self, n_ticks, write_pos, env_counter, noise_counter):
        from skillshot_learning_b200._lib import lib
        a = self.args(n_ticks, write_pos, env_counter, noise_counter)
        assert lib.ss_pool_rollout_speeds(ctypes.byref(a), None) == 0
        self.head += n_ticks

    def stepwise(self, n_ticks, write_pos, env_counter, noise_counter):
        from skillshot_learning_b200._lib import lib
        speeds, fn = self.env.speeds.data_ptr(), lib.ss_env_step_pool_speeds
        with pytest.MonkeyPatch.context() as mp:
            mp.setattr(lib, "ss_env_step_pool_blocks", lambda *a: fn(*a[:-1], speeds, a[-1]))
            super().stepwise(n_ticks, write_pos, env_counter, noise_counter)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["bf16", "f32"])
@pytest.mark.parametrize("frames,blocks,opp_frames,table,n_ticks", [(1, [40, 300, 8, 100], [1, 1, 20, 1], True, 5),
                                                                    (20, [300, 2, 62], [20, 1, 4], True, 6),
                                                                    (20, [128, 128, 128], [1, 20, 1], False, 5),
                                                                    (1, [96, 96], [20, 1], False, 6)])
def test_speeds_rollout_equals_its_stepwise_composition(precision, frames, blocks, opp_frames, table, n_ticks):
    one = _SpeedSetup(1500, blocks, frames, opp_frames, precision, 3, table=table)
    two = _SpeedSetup(1500, blocks, frames, opp_frames, precision, 3, table=table)
    L = one.L
    pos, ec, nc = L, 7, 13
    for rep in range(2):                                  # the ring wraps (3 segments, 2 x n_ticks ticks from segment 1)
        one.run(n_ticks, pos, ec, nc)
        two.stepwise(n_ticks, pos, ec, nc)
        _same(one, two)
        pos, ec, nc = (pos + n_ticks * L) % one.cap, ec + n_ticks, nc + n_ticks
    assert one.stats[:, 0].sum() > 0


# ---------------------------------------------------------------- GPU: the trainer -----------------------------------------------------
def _config5(speeds=True, **kw):
    """a 20-frame learner against 1-, 20- and 4-frame opponents, with a config-5 speed sweep"""
    from skillshot_learning_b200 import SelfPlayTrainer
    args = dict(seed=3, batch_size=1024, precision="bf16", tick_limit=40, frames=20,
                opponents=[_actor(20, scale=4.0), _actor(21, frames=20, scale=4.0), _actor(22, frames=4, scale=4.0)])
    args.update(kw)
    tr = SelfPlayTrainer(1024, **args)
    if speeds:
        tr.envs.set_speeds(*_sweep(1024, 31))
    return tr


def _calls(monkeypatch):
    """counts of the trainer's calls of ss_pool_rollout_frames and ss_pool_rollout_speeds"""
    from skillshot_learning_b200._lib import lib
    calls = dict(ss_pool_rollout_frames=0, ss_pool_rollout_speeds=0)
    for name in calls:
        def wrap(*a, _fn=getattr(lib, name), _name=name):
            calls[_name] += 1
            return _fn(*a)
        monkeypatch.setattr(lib, name, wrap)
    return calls


@pytest.mark.gpu
def test_speeds_trainer_rollout_is_its_ticks(monkeypatch):
    import torch
    calls = _calls(monkeypatch)
    t1, t2 = _config5(), _config5()
    t1.rollout(7)
    for _ in range(7):
        t2.rollout_tick()
    _same_pool(t1, t2)
    assert calls == dict(ss_pool_rollout_frames=0, ss_pool_rollout_speeds=8)
    assert sum(p["episodes"] for p in t1.pool_progress()) > 0
    # the speeds are in effect: the same trainer without them plays other games
    t3 = _config5(speeds=False)
    t3.rollout(7)
    torch.cuda.synchronize()
    assert calls == dict(ss_pool_rollout_frames=1, ss_pool_rollout_speeds=8)
    assert not torch.equal(t1.envs.state, t3.envs.state)


@pytest.mark.gpu
def test_speeds_trainer_checkpoint_resumes_bit_identically(tmp_path):
    import torch
    t1 = _config5()
    for _ in range(2):
        t1.rollout(3)
        t1.update()
    torch.save(t1.state_dict(), tmp_path / "mid.pt")
    t1.rollout(3)
    t1.update()
    blocks = t1.rebalance_pool(min_envs=4)
    torch.save(t1.state_dict(), tmp_path / "rebalanced.pt")
    for _ in range(2):
        t1.rollout(3)
        t1.update()
    # a fresh trainer without speeds, another seed and other opponents: the checkpoint brings speeds, blocks and opponents
    t2 = _config5(speeds=False, seed=8, opponents=[_actor(50), _actor(51, frames=20), _actor(52, frames=4)])
    t2.load_state_dict(torch.load(tmp_path / "rebalanced.pt", weights_only=False))
    assert t2.pool_blocks == blocks and torch.equal(t2.envs.speeds, t1.envs.speeds)
    for _ in range(2):
        t2.rollout(3)
        t2.update()
    _same_pool(t1, t2)
    assert t1.pool_blocks == t2.pool_blocks
    # from before the re-layout: the same rebalance from the same counters
    t3 = _config5(speeds=False, seed=9)
    t3.load_state_dict(torch.load(tmp_path / "mid.pt", weights_only=False))
    t3.rollout(3)
    t3.update()
    assert t3.rebalance_pool(min_envs=4) == blocks
    for _ in range(2):
        t3.rollout(3)
        t3.update()
    _same_pool(t1, t3)
