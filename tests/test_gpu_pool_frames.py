"""Training the frame-stacked learner against a pool of frozen opponents of any frame count (ss_obs_stack_push_pool,
ss_pool_rollout_frames, SelfPlayTrainer(frames=F, opponents=...)).  The GPU tests compare with ==: the fused history push
against the four launches it replaces, the one-call rollout against its stepwise composition and against ss_pool_rollout,
the pool path without pool envs against the trainer's per-tick frames loop, constant-action opponents against the C oracle,
and the trainer's checkpoint, set_opponent and evaluate_league against uninterrupted runs.  The unmarked tests run without
a GPU: argument rejection, the argument block's field order and what the trainer refuses."""
import ctypes
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _n_params(frames):
    return 12 * frames * 256 + 256 + 256 * 128 + 128 + 128 * 2 + 2


def _actor(seed, frames=1, scale=1.0):
    import torch
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(_n_params(frames), generator=g) * 0.05 * scale).float()


def _const_actor(c, frames):
    import torch
    v = torch.zeros(_n_params(frames))
    v[-2:] = torch.atanh(torch.tensor(c, dtype=torch.float32))
    return v


def _ptr(t):
    return None if t is None else t.data_ptr()


def _env_of_row(n, M):
    """learner row -> env under the pool rule (int64 [L])"""
    S = n - M
    r = np.arange(2 * S + M)
    return np.where(r < 2 * S, r // 2, r - S)


# ---------------------------------------------------------------- CPU ------------------------------------------------------------------
def _args(**kw):
    """a valid argument block (n 96, M 48, K 3 -> L 144, b 16) of fake device pointers, a 4-frame learner, opponent frames
    {1, 20, 1}, tensor cores, parameter noise in groups of 128"""
    from skillshot_learning_b200 import _lib
    Q = 4096
    a = _lib.PoolRolloutFramesArgs()
    a.state, a.n_envs, a.pool_envs, a.n_opponents, a.params, a.opp_params, a.opp_param_stride = Q, 96, 48, 3, Q, Q, 94852
    a.obs, a.act, a.reward, a.opp_obs, a.opp_act, a.done, a.winner = Q, Q, Q, Q, Q, Q, Q
    a.n_ticks, a.noise_group, a.param_noise_sd, a.tensor_cores, a.reward_mode, a.tick_limit = 4, 128, 0.5, 1, 1, 100
    a.frames, a.stack_tc, a.stack32, a.rows, a.head = 4, Q, Q, Q, 0
    frames = kw.pop("opp_frames", [1, 20, 1])
    stacks = kw.pop("opp_stacks", [None if f == 1 else Q for f in frames])
    a._keep = ((ctypes.c_int * len(frames))(*frames), (ctypes.c_void_p * len(stacks))(*stacks))
    a.opp_frames, a.opp_stacks = a._keep
    for k, v in kw.items():
        setattr(a, k, v)
    if "workspace" not in kw:
        a.workspace, a.workspace_bytes = Q, 1 << 40
    return a


def test_pool_rollout_frames_rejects_bad_arguments_without_a_gpu():
    from skillshot_learning_b200 import _lib
    L, P = _lib.lib, 4096
    assert L.ss_pool_rollout_frames(None, None) == -1
    assert L.ss_pool_rollout_frames_workspace_bytes(None) == -1
    ring = dict(ring_obs=P, ring_act=P, ring_reward=P, ring_next_obs=P, ring_done=P)
    need = L.ss_pool_rollout_frames_workspace_bytes(ctypes.byref(_args()))
    # noisy vectors: 2 groups of 144 rows x (params(4) rounded to 4) floats, then the larger layer-1 scratch (learner / opponent)
    assert need == 2 * 45700 * 4 + max(L.ss_actor_frames_tc_workspace_bytes(144, 128), L.ss_actor_frames_tc_workspace_bytes(16, 0))
    assert L.ss_pool_rollout_frames_workspace_bytes(ctypes.byref(_args(tensor_cores=0, noise_group=100))) == 2 * 45700 * 4
    assert L.ss_pool_rollout_frames_workspace_bytes(ctypes.byref(_args(frames=1, opp_frames=[1, 1, 1]))) == 0
    bad = [dict(frames=0), dict(frames=21), dict(opp_frames=[1, 0, 1]), dict(opp_frames=[1, 21, 1]),
           dict(stack_tc=None), dict(stack32=None), dict(rows=None), dict(opp_stacks=[None, None, None]),
           dict(stack32=P + 4), dict(opp_stacks=[None, P + 8, None]), dict(head=-1), dict(action_noise_sd=0.1),
           dict(workspace=None), dict(workspace=P, workspace_bytes=need - 16), dict(workspace=P + 8, workspace_bytes=need),
           dict(opp_param_stride=36484),                        # shorter than the 20-frame opponent's vector
           dict(noise_group=100), dict(noise_group=0), dict(speeds=P), dict(reward_mode=3),
           dict(n_opponents=65, pool_envs=130, n_envs=200, opp_frames=[1] * 65), dict(pool_envs=45), dict(pool_envs=50),
           dict(capacity=144 * 3 + 2, **ring), dict(capacity=144 * 3, write_pos=10, **ring), dict(capacity=144, **ring)]
    for kw in bad:
        assert L.ss_pool_rollout_frames(ctypes.byref(_args(**kw)), None) == -1, kw
    for kw in (dict(frames=0), dict(opp_frames=[1, 21, 1]), dict(noise_group=100), dict(pool_envs=50)):
        assert L.ss_pool_rollout_frames_workspace_bytes(ctypes.byref(_args(**kw))) == -1, kw
    assert L.ss_obs_stack_push_pool(P, P, 96, 48, 21, 0, P, None, P, None, None) == -1
    assert L.ss_obs_stack_push_pool(P, None, 96, 48, 4, 0, P, None, P, None, None) == -1
    assert L.ss_obs_stack_push_pool(P, P, 96, 97, 4, 0, P, None, P, None, None) == -1
    assert L.ss_obs_stack_push_pool(P, P, 96, 48, 4, 0, P, None, P, P + 4, None) == -1


def test_pool_frames_argument_block_matches_the_header():
    """The ctypes mirror of struct ss_pool_rollout_frames_args lists the header's fields in the header's order."""
    from skillshot_learning_b200 import _lib
    text = open(os.path.join(ROOT, "include", "skillshot_b200.h")).read()
    body = re.search(r"typedef struct ss_pool_rollout_frames_args \{(.*?)\} ss_pool_rollout_frames_args;", text, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = []
    for decl in body.split(";"):
        decl = decl.strip()
        if decl:
            names += [re.sub(r"[\s\*]|const", "", part.split()[-1]) for part in decl.split(",")]
    assert names == [f[0] for f in _lib.PoolRolloutFramesArgs._fields_]


def test_frame_stacked_pool_trainer_rejects_what_it_cannot_run_without_a_gpu():
    from skillshot_learning_b200 import SelfPlayTrainer
    opp = [_actor(1), _actor(2, frames=20)]
    for kw in (dict(process_group=object()), dict(reward_mode="simple"), dict(precision="bf16", noise_group=100)):
        with pytest.raises(ValueError):
            SelfPlayTrainer(64, frames=4, opponents=opp, **kw)
    with pytest.raises(ValueError):
        SelfPlayTrainer(64, frames=4, opponents=[_actor(1), np.zeros(100)])        # no actor's parameter count
    # the pool's replay-capacity rule (3 opponents: 30 pool envs, L = 2 * 64 - 30 = 98 learner rows): a multiple of L, at
    # least two of them
    for cap in (1000, 98, 100):
        with pytest.raises(ValueError, match="replay capacity"):
            SelfPlayTrainer(64, device="cuda", frames=4, opponents=[_actor(1), _actor(2, frames=20), _actor(3)], replay_capacity=cap)


def test_frame_stacked_learners_and_opponents_pass_the_pool_rules_without_a_gpu():
    """A frame-stacked learner and multi-frame opponents are accepted by every rule of the pool: without a CUDA device the
    construction gets as far as the envs, which need one."""
    import torch
    from skillshot_learning_b200 import SelfPlayTrainer
    cases = (dict(frames=2, opponents=[_actor(1)] * 3), dict(opponents=[_actor(1), _actor(2, frames=2)]),
             dict(frames=20, opponents=[_actor(1, frames=20), _actor(2, frames=4)], replay_capacity=4 * (2 * 64 - 32)))
    for kw in cases:
        if torch.cuda.is_available():
            tr = SelfPlayTrainer(64, device="cuda", **kw)
            assert tr.opp_frames == [int(round((v.numel() - 33410) / 3072)) for v in kw["opponents"]]
        else:
            with pytest.raises(RuntimeError, match="CUDA device"):
                SelfPlayTrainer(64, device="cuda", **kw)


# ---------------------------------------------------------------- GPU: the push kernel -------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("frames", [1, 4, 20])
@pytest.mark.parametrize("n,M", [(300, 0), (1000, 384)])          # 2S = 600 and 1232: not multiples of 128
def test_push_pool_equals_the_composition_it_replaces(frames, n, M):
    import torch
    from skillshot_learning_b200._lib import lib
    S, L = n - M, 2 * n - M
    env = torch.from_numpy(_env_of_row(n, M)).cuda()
    d = dict(device="cuda")
    tc_bytes = lib.ss_obs_stack_tc_bytes(L, frames)
    ref = dict(tc=torch.zeros(tc_bytes, dtype=torch.uint8, **d), s32=torch.zeros(L, frames, 12, **d), rows=torch.zeros(L, 12 * frames, **d))
    new = dict(tc=torch.zeros(tc_bytes, dtype=torch.uint8, **d), s32=torch.zeros(L, frames, 12, **d), rows=torch.zeros(L, 12 * frames, **d),
               rows2=torch.zeros(L, 12 * frames, **d))
    ring = dict(obs=torch.zeros(2 * L, 12 * frames, **d), act=torch.zeros(2 * L, 2, **d), reward=torch.zeros(2 * L, **d),
                next_obs=torch.zeros(2 * L, 12 * frames, **d), done=torch.zeros(2 * L, dtype=torch.uint8, **d))
    act, rew = torch.zeros(L, 2, **d), torch.zeros(L, **d)
    g = torch.Generator(device="cuda").manual_seed(frames)
    for head in range(0, 2 * frames + 3):
        obs = torch.randn(L, 12, generator=g, **d)
        done = (torch.rand(n, generator=g, **d) < 0.15).to(torch.uint8) if head else torch.ones(n, dtype=torch.uint8, **d)
        if head:
            done[S:S + 3], done[n - 3:] = 1, 1                # pool restarts with the learner in seat 1 and in seat 2
        done_rows = done[env].contiguous()
        prev = ref["rows"].clone()
        assert lib.ss_obs_stack_push_tc(ref["tc"].data_ptr(), L, frames, head, obs.data_ptr(), done_rows.data_ptr(), 1, None) == 0
        assert lib.ss_obs_stack_push(ref["s32"].data_ptr(), L, frames, head, obs.data_ptr(), done_rows.data_ptr(), 1, None) == 0
        assert lib.ss_obs_stack_ordered(ref["s32"].data_ptr(), L, frames, head, ref["rows"].data_ptr(), None) == 0
        assert lib.ss_replay_push_frames(ring["obs"].data_ptr(), ring["act"].data_ptr(), ring["reward"].data_ptr(),
                                         ring["next_obs"].data_ptr(), ring["done"].data_ptr(), 2 * L, 0, frames, prev.data_ptr(),
                                         act.data_ptr(), rew.data_ptr(), ref["rows"].data_ptr(), None, 1, L, None) == 0
        assert lib.ss_obs_stack_push_pool(new["tc"].data_ptr(), new["s32"].data_ptr(), n, M, frames, head, obs.data_ptr(),
                                          done.data_ptr(), new["rows"].data_ptr(), new["rows2"].data_ptr(), None) == 0
        torch.cuda.synchronize()
        for k in ("tc", "s32", "rows"):
            assert torch.equal(ref[k], new[k]), (k, head)
        assert torch.equal(new["rows2"], new["rows"])
        assert torch.equal(ring["next_obs"][:L], new["rows"]) and torch.equal(ring["obs"][:L], prev)
    # the float32 history alone (stack_tc NULL), without a second output
    s32 = torch.zeros(L, frames, 12, **d)
    rows = torch.zeros(L, 12 * frames, **d)
    obs = torch.randn(L, 12, generator=g, **d)
    assert lib.ss_obs_stack_push_pool(None, s32.data_ptr(), n, M, frames, 0, obs.data_ptr(), None, rows.data_ptr(), None, None) == 0
    torch.cuda.synchronize()
    assert torch.equal(s32[:, 0], obs) and torch.equal(rows[:, 12 * (frames - 1):], obs)


# ---------------------------------------------------------------- GPU: the rollout -----------------------------------------------------
class _Setup:
    """Device buffers of one pool rollout: n envs, M pool envs, the learner's frames and the opponents' frames."""

    def __init__(self, n, M, frames, opp_frames, precision, segs, seed=5):
        import torch
        from skillshot_learning_b200 import SkillshotEnvs
        from skillshot_learning_b200._lib import lib
        from skillshot_learning_b200.learner import pool_layout
        d = dict(device="cuda")
        K = len(opp_frames)
        self.n, self.M, self.K, self.L, self.S = n, M, K, 2 * n - M, n - M
        self.b = M // K if M else 0
        self.F, self.opp_frames, self.tc = frames, list(opp_frames), 1 if precision == "bf16" else 0
        L, b = self.L, self.b
        self.env = SkillshotEnvs(n, random_positions=True, seed=seed)
        rows = torch.from_numpy(pool_layout(n, M, K).reshape(-1)).cuda()
        self.obs = torch.empty(2 * n, 12, **d)
        self.obs[rows] = self.env.observe().reshape(-1, 12)
        self.stride = max((_n_params(f) + 3) // 4 * 4 for f in opp_frames)
        self.opp = torch.zeros(K, self.stride, **d)
        for k, f in enumerate(opp_frames):
            self.opp[k, :_n_params(f)] = _actor(40 + k, frames=f, scale=4.0).cuda()
        self.params = _actor(9, frames=frames, scale=3.0).cuda()
        self.head = 0
        self.stack_tc = self.stack32 = self.rows = None
        if frames > 1:
            self.stack32 = torch.zeros(L, frames, 12, **d)
            self.stack_tc = torch.zeros(lib.ss_obs_stack_tc_bytes(L, frames), dtype=torch.uint8, **d) if self.tc else None
            self.rows = torch.zeros(L, 12 * frames, **d)
            assert lib.ss_obs_stack_push_pool(_ptr(self.stack_tc), self.stack32.data_ptr(), n, M, frames, 0, self.obs.data_ptr(),
                                              torch.ones(n, dtype=torch.uint8, **d).data_ptr(), self.rows.data_ptr(), None, None) == 0
        self.opp_stacks = []
        for k, f in enumerate(opp_frames):
            if f == 1 or not M:
                self.opp_stacks.append(None)
                continue
            s = (torch.zeros(lib.ss_obs_stack_tc_bytes(b, f), dtype=torch.uint8, **d) if self.tc else torch.zeros(b, f, 12, **d))
            push = lib.ss_obs_stack_push_tc if self.tc else lib.ss_obs_stack_push
            assert push(s.data_ptr(), b, f, 0, self.obs[L + k * b:].data_ptr(), None, 1, None) == 0
            self.opp_stacks.append(s)
        self.cap = segs * L
        w = 12 * frames
        self.ring = dict(obs=torch.zeros(self.cap, w, **d), act=torch.zeros(self.cap, 2, **d), reward=torch.zeros(self.cap, **d),
                         next_obs=torch.zeros(self.cap, w, **d), done=torch.zeros(self.cap, dtype=torch.uint8, **d))
        self.status = torch.zeros(2 + 144, dtype=torch.int32, **d)
        self.stats = torch.zeros(max(K, 1), 8, dtype=torch.int64, **d)
        self.act = torch.zeros(2 * n, 2, **d)
        self.reward = torch.zeros(L, **d)
        self.done = torch.zeros(n, dtype=torch.uint8, **d)
        self.winner = torch.zeros(n, dtype=torch.uint8, **d)
        self.ws = None

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
        if r is not None:
            a.ring_obs, a.ring_act, a.ring_reward, a.ring_next_obs, a.ring_done = (r[k].data_ptr() for k in ("obs", "act", "reward", "next_obs", "done"))
            a.capacity, a.write_pos = self.cap, write_pos
        a.n_ticks = n_ticks
        a.param_noise_sd, a.noise_group, a.tensor_cores, a.reward_mode, a.tick_limit = 0.5, 128, self.tc, 1, 60
        a.reset_mode, a.env_seed, a.env_counter, a.noise_seed, a.noise_counter = 1, 5, env_counter, 11, noise_counter
        a.status, a.step_flags, a.pool_stats = self.status.data_ptr(), 2, self.stats.data_ptr()
        a.frames, a.stack_tc, a.stack32, a.rows, a.head = self.F, _ptr(self.stack_tc), _ptr(self.stack32), _ptr(self.rows), self.head
        a._keep = ((ctypes.c_int * self.K)(*self.opp_frames), (ctypes.c_void_p * self.K)(*[_ptr(s) for s in self.opp_stacks]))
        a.opp_frames, a.opp_stacks = a._keep
        need = _lib.lib.ss_pool_rollout_frames_workspace_bytes(ctypes.byref(a))
        assert need >= 0
        if need:
            self.ws = torch.zeros(need, dtype=torch.uint8, device="cuda")
            a.workspace, a.workspace_bytes = self.ws.data_ptr(), need
        return a

    def run(self, n_ticks, write_pos, env_counter, noise_counter):
        from skillshot_learning_b200._lib import lib
        a = self.args(n_ticks, write_pos, env_counter, noise_counter)
        assert lib.ss_pool_rollout_frames(ctypes.byref(a), None) == 0
        self.head += n_ticks

    def stepwise(self, n_ticks, write_pos, env_counter, noise_counter):
        """ss_pool_rollout_frames composed from the existing entry points, tick by tick (the learner's history step as
        ss_obs_stack_push_tc, ss_obs_stack_push and ss_obs_stack_ordered with per-row restart flags)"""
        import torch
        from skillshot_learning_b200._lib import lib
        n, M, K, L, b, F, r = self.n, self.M, self.K, self.L, self.b, self.F, self.ring
        ring = r is not None
        segs = self.cap // L if ring else 1
        seg = write_pos // L if ring else 0
        if ring:
            r["obs"][seg * L:(seg + 1) * L] = self.rows if F > 1 else self.obs[:L]
        env = torch.from_numpy(_env_of_row(n, M)).cuda()
        stride = (_n_params(F) + 3) // 4 * 4
        groups = (L + 127) // 128
        noisy = torch.zeros(groups * stride, device="cuda")
        ws = torch.zeros(max(lib.ss_actor_frames_tc_workspace_bytes(L, 128), lib.ss_actor_frames_tc_workspace_bytes(max(b, 1), 0)),
                         dtype=torch.uint8, device="cuda")
        seg_rows = (ctypes.c_int64 * K)(*([b] * K))
        oo, oa = self.obs[L:], self.act[L:]
        for t in range(n_ticks):
            head = self.head + t
            last = t + 1 == n_ticks
            nxt = (seg + 1) % segs
            o = r["obs"][seg * L:(seg + 1) * L] if ring else self.obs[:L]
            a = r["act"][seg * L:(seg + 1) * L] if ring else self.act[:L]
            if F > 1:
                assert lib.ss_param_noise_groups(self.params.data_ptr(), noisy.data_ptr(), _n_params(F), groups, stride, 0.5, 11,
                                                 noise_counter + t, None) == 0
                if self.tc:
                    assert lib.ss_actor_forward_frames_tc(noisy.data_ptr(), stride, 128, self.stack_tc.data_ptr(), F, head, a.data_ptr(), L,
                                                          ws.data_ptr(), ws.numel(), None) == 0
                else:
                    assert lib.ss_actor_forward_frames(noisy.data_ptr(), stride, 128, self.stack32.data_ptr(), F, head, a.data_ptr(), L,
                                                       None) == 0
            else:
                fwd = lib.ss_actor_forward_tc if self.tc else lib.ss_actor_forward
                assert fwd(self.params.data_ptr(), o.data_ptr(), a.data_ptr(), L, 0.5, 128, 0.0, 11, noise_counter + t, None) == 0
            k = 0
            while M and k < K:
                f = self.opp_frames[k]
                p = self.opp[k].data_ptr()
                if f > 1:
                    if self.tc:
                        assert lib.ss_actor_forward_frames_tc(p, 0, 0, self.opp_stacks[k].data_ptr(), f, head, oa[k * b:].data_ptr(), b,
                                                              ws.data_ptr(), ws.numel(), None) == 0
                    else:
                        assert lib.ss_actor_forward_frames(p, 0, 0, self.opp_stacks[k].data_ptr(), f, head, oa[k * b:].data_ptr(), b,
                                                           None) == 0
                    k += 1
                elif self.tc:
                    e = k + 1
                    while e < K and self.opp_frames[e] == 1:
                        e += 1
                    rows = (ctypes.c_int64 * (e - k))(*([b] * (e - k)))
                    assert lib.ss_actor_forward_segments_tc(p, self.stride, rows, e - k, oo[k * b:].data_ptr(), oa[k * b:].data_ptr(),
                                                            None) == 0
                    k = e
                else:
                    assert lib.ss_actor_forward(p, oo[k * b:].data_ptr(), oa[k * b:].data_ptr(), b, 0.0, 1, 0.0, 0, 0, None) == 0
                    k += 1
            if F > 1:
                obs_out, obs2 = self.obs[:L], None
            elif ring:
                obs_out = r["next_obs"][seg * L:(seg + 1) * L]
                obs2 = r["obs"][nxt * L:(nxt + 1) * L] if not last else self.obs[:L]
            else:
                obs_out, obs2 = self.obs[:L], None
            assert lib.ss_env_step_pool(self.env.state.data_ptr(), n, M, K, a.data_ptr(), oa.data_ptr() if M else None, obs_out.data_ptr(),
                                        _ptr(obs2), (r["reward"][seg * L:] if ring else self.reward).data_ptr(),
                                        r["done"][seg * L:].data_ptr() if ring else None, oo.data_ptr() if M else None,
                                        self.done.data_ptr(), self.winner.data_ptr(), 1, 60, 1, 5, env_counter + t,
                                        self.status.data_ptr(), 2, self.stats.data_ptr(), None) == 0
            if F > 1:
                done_rows = self.done[env].contiguous()
                if self.tc:
                    assert lib.ss_obs_stack_push_tc(self.stack_tc.data_ptr(), L, F, head + 1, self.obs.data_ptr(), done_rows.data_ptr(), 1,
                                                    None) == 0
                assert lib.ss_obs_stack_push(self.stack32.data_ptr(), L, F, head + 1, self.obs.data_ptr(), done_rows.data_ptr(), 1, None) == 0
                assert lib.ss_obs_stack_ordered(self.stack32.data_ptr(), L, F, head + 1, self.rows.data_ptr(), None) == 0
                if ring:
                    r["next_obs"][seg * L:(seg + 1) * L] = self.rows
                    if not last:
                        r["obs"][nxt * L:(nxt + 1) * L] = self.rows
            for k, f in enumerate(self.opp_frames):
                if f == 1 or not M:
                    continue
                push = lib.ss_obs_stack_push_tc if self.tc else lib.ss_obs_stack_push
                assert push(self.opp_stacks[k].data_ptr(), b, f, head + 1, oo[k * b:].data_ptr(), self.done[self.S + k * b:].data_ptr(), 1,
                            None) == 0
            seg = nxt
        if ring:
            last = (seg + segs - 1) % segs
            self.act[:L] = r["act"][last * L:(last + 1) * L]
            self.reward.copy_(r["reward"][last * L:(last + 1) * L])
        self.head += n_ticks
        torch.cuda.synchronize()


def _same(s1, s2):
    import torch
    torch.cuda.synchronize()
    for k in ("obs", "act", "reward", "done", "winner", "status", "stats", "stack_tc", "stack32", "rows"):
        a, b = getattr(s1, k), getattr(s2, k)
        assert (a is None and b is None) or torch.equal(a, b), k
    assert torch.equal(s1.env.state, s2.env.state)
    for a, b in zip(s1.opp_stacks, s2.opp_stacks):
        assert (a is None and b is None) or torch.equal(a, b), "opponent history"
    for k in s1.ring or {}:
        assert torch.equal(s1.ring[k], s2.ring[k]), k
    assert s1.head == s2.head


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["bf16", "f32"])
@pytest.mark.parametrize("n_ticks", [5, 6])
@pytest.mark.parametrize("frames,opp_frames", [(4, [1, 1, 1]), (20, [20, 20]), (20, [1, 20, 4, 1]), (1, [20, 1])])
def test_pool_rollout_frames_equals_its_stepwise_composition(precision, n_ticks, frames, opp_frames):
    n, M = 1500, 96 * len(opp_frames)
    one, two = _Setup(n, M, frames, opp_frames, precision, 3), _Setup(n, M, frames, opp_frames, precision, 3)
    L = one.L
    pos, ec, nc = L, 7, 13
    for rep in range(2):                                  # the ring wraps (3 segments, 2 x n_ticks ticks from segment 1)
        one.run(n_ticks, pos, ec, nc)
        two.stepwise(n_ticks, pos, ec, nc)
        _same(one, two)
        pos, ec, nc = (pos + n_ticks * L) % one.cap, ec + n_ticks, nc + n_ticks
    assert one.stats[:, 0].sum() > 0
    # without a ring the learner's rows are rewritten in place
    one.ring = two.ring = None
    one.run(3, 0, ec, nc)
    two.stepwise(3, 0, ec, nc)
    _same(one, two)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["bf16", "f32"])
def test_all_one_frame_pool_rollout_frames_is_the_pool_rollout(precision):
    from skillshot_learning_b200 import _lib
    n, M, K, T = 2560, 1536, 6, 5
    one, two = _Setup(n, M, 1, [1] * K, precision, 3), _Setup(n, M, 1, [1] * K, precision, 3)
    a = one.args(T, one.L, 7, 13)
    assert _lib.lib.ss_pool_rollout_frames(ctypes.byref(a), None) == 0
    one.head += T
    f = two.args(T, two.L, 7, 13)
    p = _lib.PoolRolloutArgs()
    for name, _ in _lib.PoolRolloutArgs._fields_:
        setattr(p, name, getattr(f, name))
    assert _lib.lib.ss_pool_rollout(ctypes.byref(p), None) == 0
    two.head += T
    _same(one, two)


def _trainer(**kw):
    from skillshot_learning_b200 import SelfPlayTrainer
    args = dict(seed=3, batch_size=1024, precision="bf16", tick_limit=40, frames=4)
    args.update(kw)
    return SelfPlayTrainer(1024, **args)


def _same_trainer(t1, t2):
    import torch
    torch.cuda.synchronize()
    assert torch.equal(t1.networks.params, t2.networks.params) and torch.equal(t1.networks.target, t2.networks.target)
    assert torch.equal(t1.envs.state, t2.envs.state)
    for k in ("obs", "act", "reward", "next_obs", "done"):
        assert torch.equal(getattr(t1.replay, k), getattr(t2.replay, k)), k
    assert torch.equal(t1.stack.stack, t2.stack.stack) and torch.equal(t1.rows, t2.rows)
    assert (t1.stack.stack32 is None) == (t2.stack.stack32 is None)
    if t1.stack.stack32 is not None:
        assert torch.equal(t1.stack.stack32, t2.stack.stack32)
    assert t1.stack.head == t2.stack.head and t1.stack.counter == t2.stack.counter
    assert t1.envs.counter == t2.envs.counter and t1.networks.counter == t2.networks.counter
    assert t1.replay.pos == t2.replay.pos and t1.replay.size == t2.replay.size


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["bf16", "f32"])
def test_without_pool_envs_the_pool_path_is_the_frames_loop(precision):
    import torch
    ref = _trainer(precision=precision, tick_limit=5)          # every game restarts at least once in 11 ticks
    pool = _trainer(precision=precision, tick_limit=5, opponents=[_actor(1, frames=20)], pool_envs=0)
    for _ in range(11):
        ref.rollout_tick()
    pool.rollout(5)
    pool.rollout(6)
    _same_trainer(ref, pool)
    assert torch.equal(ref.obs.reshape(-1, 12), pool.obs)


@pytest.mark.gpu
def test_stored_rows_are_consistent():
    """Every learner row's next observation is its observation shifted by one frame, and after an episode end (hit or tick
    limit) every frame is the restarted game's first observation."""
    import torch
    tr = _trainer(opponents=[_actor(1), _actor(2, frames=20)], pool_envs=512, tick_limit=12)
    L, F = tr.learner_rows, tr.frames
    env = torch.from_numpy(_env_of_row(1024, 512)).cuda()
    restarts = 0
    for t in range(30):
        out = tr.rollout_tick()
        p = (tr.replay.pos - L) % tr.replay.capacity
        obs, nxt = tr.replay.obs[p:p + L].view(L, F, 12), tr.replay.next_obs[p:p + L].view(L, F, 12)
        done = out["done"][env].bool()
        assert torch.equal(nxt[~done, :-1], obs[~done, 1:])
        assert torch.equal(nxt[done], nxt[done, -1:].expand(-1, F, -1).contiguous())
        assert torch.equal(nxt[:, -1], tr.obs[:L])
        assert torch.equal(tr.rows, nxt.reshape(L, -1))
        restarts += int(done.sum())
    assert restarts > 0


@pytest.mark.gpu
def test_constant_action_frame_stacked_opponents_equal_the_oracle():
    """A 20-frame and a 1-frame opponent with zero weights and constant output biases: the learner's actions read back from
    the ring and the opponents' constant actions replayed through the C oracle give the same positions, winners, rewards and
    hit flags."""
    import torch
    from oracle.oracle import OracleEnvs
    from skillshot_learning_b200.learner import pool_layout
    n, M, T = 800, 512, 40
    consts = [((0.898, -0.08), 20), ((0.189, -0.324), 1)]
    s = _Setup(n, M, 4, [f for _, f in consts], "bf16", T + 1)
    L, S, K = s.L, s.S, len(consts)
    s.env.reset(random_positions=False)
    from skillshot_learning_b200._lib import lib
    rows = torch.from_numpy(pool_layout(n, M, K).reshape(-1)).cuda()
    s.obs[rows] = s.env.observe().reshape(-1, 12)
    # every history restarted from the reset observations
    ones = torch.ones(n, dtype=torch.uint8, device="cuda")
    assert lib.ss_obs_stack_push_pool(s.stack_tc.data_ptr(), s.stack32.data_ptr(), n, M, 4, 0, s.obs.data_ptr(), ones.data_ptr(),
                                      s.rows.data_ptr(), None, None) == 0
    assert lib.ss_obs_stack_push_tc(s.opp_stacks[0].data_ptr(), s.b, 20, 0, s.obs[L:].data_ptr(), ones.data_ptr(), 1, None) == 0
    for k, (c, f) in enumerate(consts):
        s.opp[k].zero_()
        s.opp[k, :_n_params(f)] = _const_actor(c, f).cuda()
    a = s.args(T, 0, 0, 0)
    a.reward_mode, a.reset_mode, a.tick_limit = 2, 0, 25
    assert lib.ss_pool_rollout_frames(ctypes.byref(a), None) == 0
    torch.cuda.synchronize()
    opp_act = s.act[L:].cpu().numpy()
    assert all((opp_act[k * s.b:(k + 1) * s.b] == opp_act[k * s.b]).all() for k in range(K))
    ring = {k: v.cpu().numpy() for k, v in s.ring.items()}
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
    want, got = orc.snapshot(), s.env.export_state()
    for k in ("px", "py", "qx", "qy", "ticks", "live", "winner"):
        assert np.array_equal(got[k], want[k]), k
    assert s.stats[:, 0].sum() > 0 and S > 0


def _mixed(**kw):
    return _trainer(opponents=[_actor(20, scale=4.0), _actor(21, frames=20, scale=4.0), _actor(22, frames=4, scale=4.0)], **kw)


def _same_pool(t1, t2):
    import torch
    _same_trainer(t1, t2)
    assert torch.equal(t1.obs, t2.obs) and torch.equal(t1.pool_stats, t2.pool_stats) and torch.equal(t1.opponents, t2.opponents)
    assert t1.pool_head == t2.pool_head
    for a, b in zip(t1.opp_stacks, t2.opp_stacks):
        assert (a is None and b is None) or torch.equal(a, b)


@pytest.mark.gpu
def test_frame_stacked_pool_trainer_checkpoint_resumes_bit_identically():
    import torch
    t1 = _mixed()
    assert t1.pool_envs == 510 and t1.opponents.shape[1] == 94852 and t1.opp_frames == [1, 20, 4]
    assert t1.rows.shape == (t1.learner_rows, 48)
    for _ in range(3):
        t1.rollout(3)
        t1.update()
    torch.cuda.synchronize()
    sd = t1.state_dict()
    for _ in range(3):
        t1.rollout(3)
        t1.update()
    t2 = _trainer(seed=8, opponents=[_actor(50), _actor(51, frames=20), _actor(52, frames=4)])
    t2.load_state_dict(sd)
    for _ in range(3):
        t2.rollout(3)
        t2.update()
    _same_pool(t1, t2)
    prog = t1.pool_progress()
    assert len(prog) == 3 and sum(p["episodes"] for p in prog) > 0
    for other in (dict(opponents=[_actor(1), _actor(2, frames=20), _actor(3, frames=20)]),      # another opponent's frames
                  dict(opponents=[_actor(1), _actor(2, frames=20), _actor(3, frames=4)], frames=5),
                  dict(opponents=[_actor(1), _actor(2, frames=20)]), dict(opponents=None)):
        with pytest.raises(ValueError):
            _trainer(**other).load_state_dict(sd)
    # a 1-frame learner against a 20-frame opponent: the opponent's history and the pool's slot counter come back
    v1 = _trainer(frames=1, opponents=[_actor(1), _actor(2, frames=20)])
    v1.rollout(3)
    sd1 = v1.state_dict()
    v1.rollout(4)
    v2 = _trainer(frames=1, seed=9, opponents=[_actor(3), _actor(4, frames=20)])
    v2.load_state_dict(sd1)
    v2.rollout(4)
    torch.cuda.synchronize()
    assert v1.pool_head == v2.pool_head == 7 and torch.equal(v1.envs.state, v2.envs.state)
    assert torch.equal(v1.opp_stacks[1], v2.opp_stacks[1]) and torch.equal(v1.replay.obs, v2.replay.obs)
    # a checkpoint of a pool of 1-frame actors written without frame counts and histories still loads into a 1-frame trainer
    u1 = _trainer(frames=1, opponents=[_actor(1), _actor(2)])
    u1.rollout(3)
    old = u1.state_dict()
    for k in ("frames", "stacks", "head"):
        del old["pool"][k]
    u2 = _trainer(frames=1, seed=9, opponents=[_actor(3), _actor(4)])
    u2.load_state_dict(old)
    u1.rollout(2)
    u2.rollout(2)
    torch.cuda.synchronize()
    assert torch.equal(u1.envs.state, u2.envs.state) and torch.equal(u1.replay.obs, u2.replay.obs)


@pytest.mark.gpu
def test_set_opponent_on_a_frame_stacked_slot_takes_effect_on_the_next_tick():
    import torch
    new = _actor(77, frames=20, scale=4.0)
    t1, t2, t3 = _mixed(), _mixed(), _mixed()
    t1.rollout(4)
    t1.set_opponent(1, new)
    t1.rollout(5)
    for _ in range(4):
        t2.rollout_tick()
    shapes = [(240, 256), (256,), (256, 128), (128,), (128, 2), (2,)]
    parts, o = [], 0
    for sh in shapes:
        k = int(np.prod(sh))
        parts.append(new[o:o + k].reshape(sh).numpy())
        o += k
    t2.set_opponent(1, parts)
    for _ in range(5):
        t2.rollout_tick()
    t3.rollout(9)
    _same_pool(t1, t2)
    assert not torch.equal(t1.envs.state, t3.envs.state)
    for k, actor in ((1, _actor(5)), (0, _actor(5, frames=20)), (2, _actor(5, frames=20))):
        with pytest.raises(ValueError):
            t1.set_opponent(k, actor)


@pytest.mark.gpu
def test_evaluate_league_does_not_disturb_frame_stacked_pool_training():
    def run(evaluate):
        tr = _mixed()
        for k in range(4):
            tr.rollout(4)
            tr.update()
            if evaluate and k == 1:
                tr.evaluate_league([_actor(90), _actor(91, frames=20)], games_per_pair=512, seed=2, tick_limit=100)
        return tr
    _same_pool(run(True), run(False))
