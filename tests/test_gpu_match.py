"""Matches between two actors (ss_env_step_match, ss_actor_forward_groups_tc, ss_match_summary, ss_match_play, Match,
SelfPlayTrainer.evaluate).  The GPU tests compare with ==: the seat-mapped step against ss_env_step under the seat
permutation, the grouped forward against ss_actor_forward_tc per group, the summary against a host tally, the one-call
match against its stepwise composition, and constant-action games against the C oracle.  The unmarked tests run without a
GPU: argument rejection, workspace sizes, the argument block's field order, actor parsing and the result arithmetic."""
import ctypes
import math
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
A_N = 36482
STRIDE = 36484


# ---------------------------------------------------------------- helpers --------------------------------------------------------------
def _host_tally(ticks, live, winner, split, tick_limit):
    """[2][8] counters of ss_match_summary from exported state (block 0: A is player 1, winner_id = the player HIT)."""
    out = np.zeros((2, 8), np.int64)
    for blk, sl in ((0, slice(0, split)), (1, slice(split, None))):
        t, lv, w = ticks[sl], live[sl], winner[sl]
        a_hit = w == blk + 1
        out[blk, 0] = t.size
        out[blk, 1] = int(((lv == 0) & ~a_hit).sum())
        out[blk, 2] = int(((lv == 0) & a_hit).sum())
        out[blk, 3] = int(((lv != 0) & (t >= tick_limit)).sum())
        out[blk, 4] = int(((lv != 0) & (t < tick_limit)).sum())
        out[blk, 5] = int(t[lv == 0].sum())
    return out


def _seat_actions(act_pm, split):
    """policy-major [2][n][2] -> per-env [n][2 players][2]"""
    import torch
    n = act_pm.shape[1]
    a_first = (torch.arange(n, device=act_pm.device) < split)[:, None]
    p1 = torch.where(a_first, act_pm[0], act_pm[1])
    p2 = torch.where(a_first, act_pm[1], act_pm[0])
    return torch.stack([p1, p2], dim=1).contiguous()


def _seat_obs(obs, split):
    """per-env [n][2][12] -> policy-major [2][n][12]"""
    import torch
    n = obs.shape[0]
    a_first = (torch.arange(n, device=obs.device) < split)[:, None]
    return torch.stack([torch.where(a_first, obs[:, 0], obs[:, 1]), torch.where(a_first, obs[:, 1], obs[:, 0])]).contiguous()


def _actor(frames, seed, scale=1.0):
    import torch
    from skillshot_learning_b200 import _lib
    n = int(_lib.lib.ss_actor_frames_params(frames))
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(n, generator=g) * 0.05 * scale).float()


def _speeds(n, seed):
    rng = np.random.default_rng(seed)
    return (rng.uniform(1.0, 5.0, n), rng.uniform(0.05, 0.5, n), rng.uniform(2.0, 8.0, n), rng.integers(5, 30, n))


# ---------------------------------------------------------------- CPU ------------------------------------------------------------------
def test_match_entry_points_reject_bad_arguments_without_a_gpu():
    from skillshot_learning_b200 import _lib
    L = _lib.lib
    P, Q = 4096, 4097                      # aligned / misaligned fake device pointers, never dereferenced
    assert L.ss_env_step_match(None, 16, 8, P, P, 100, None, None, None) == -1
    assert L.ss_env_step_match(P, 16, 8, None, P, 100, None, None, None) == -1
    assert L.ss_env_step_match(P, 16, 17, P, P, 100, None, None, None) == -1          # split > n
    assert L.ss_env_step_match(P, 16, -1, P, P, 100, None, None, None) == -1
    assert L.ss_env_step_match(P, 16, 8, P, P, 0, None, None, None) == -1             # tick_limit <= 0
    assert L.ss_env_step_match(P, 0, 0, P, P, 100, None, None, None) == -1
    assert L.ss_env_step_match(Q, 16, 8, P, P, 100, None, None, None) == -1
    assert L.ss_env_step_match(P, 16, 8, P + 4, P, 100, None, None, None) == -1
    assert L.ss_env_step_match(P, 16, 8, P, P + 8, 100, None, None, None) == -1
    assert L.ss_env_step_match(P, 16, 8, P, P, 100, P + 8, None, None) == -1
    assert L.ss_actor_forward_groups_tc(None, STRIDE, 8, P, P, 16, None) == -1
    assert L.ss_actor_forward_groups_tc(P, STRIDE, 0, P, P, 16, None) == -1
    assert L.ss_actor_forward_groups_tc(P, STRIDE, 8, P, P, 0, None) == -1
    assert L.ss_actor_forward_groups_tc(P, STRIDE + 2, 8, P, P, 16, None) == -1       # stride not a multiple of 4
    assert L.ss_actor_forward_groups_tc(P, 1024, 8, P, P, 16, None) == -1             # vectors would overlap
    assert L.ss_actor_forward_groups_tc(P, -4, 8, P, P, 16, None) == -1
    assert L.ss_actor_forward_groups_tc(P + 4, STRIDE, 8, P, P, 16, None) == -1
    assert L.ss_actor_forward_groups_tc(P, STRIDE, 8, P + 4, P, 16, None) == -1
    assert L.ss_actor_forward_groups_tc(P, STRIDE, 8, P, P + 4, 16, None) == -1
    assert L.ss_match_summary(None, 16, 8, 100, P, None) == -1
    assert L.ss_match_summary(P, 16, 8, 100, None, None) == -1
    assert L.ss_match_summary(P, 16, 20, 100, P, None) == -1
    assert L.ss_match_summary(P, 16, 8, 0, P, None) == -1
    assert L.ss_match_summary(P + 8, 16, 8, 100, P, None) == -1
    assert L.ss_match_summary(P, 16, 8, 100, P + 4, None) == -1
    assert L.ss_match_play(None, None) == -1

    def args(**kw):
        a = _lib.MatchArgs()
        a.state, a.n_envs, a.split, a.tick_limit = P, 256, 100, 50
        a.obs, a.act, a.params, a.param_stride = P, P, P, STRIDE
        a.frames_a = a.frames_b = 1
        a.head, a.tensor_cores, a.n_ticks = 0, 1, 4
        for k, v in kw.items():
            setattr(a, k, v)
        return a
    f20 = int(L.ss_actor_frames_params(20))
    ws = int(L.ss_match_workspace_bytes(256, 20, 1, 1))
    bad = [dict(state=None), dict(obs=None), dict(act=None), dict(params=None), dict(state=Q), dict(obs=P + 8), dict(act=P + 4),
           dict(params=P + 4), dict(speeds=P + 8), dict(status=P + 2), dict(n_envs=0), dict(split=-1), dict(split=257),
           dict(tick_limit=0), dict(frames_a=0), dict(frames_b=21), dict(param_stride=STRIDE - 4), dict(param_stride=STRIDE + 2),
           dict(n_ticks=0), dict(head=-1),
           dict(frames_a=20, param_stride=(f20 + 3) // 4 * 4, stack_a=None, workspace=P, workspace_bytes=ws),        # no history
           dict(frames_a=20, param_stride=STRIDE, stack_a=P, workspace=P, workspace_bytes=ws),                        # short stride
           dict(frames_a=20, param_stride=(f20 + 3) // 4 * 4, stack_a=P, workspace=P, workspace_bytes=ws - 1),        # short workspace
           dict(frames_a=20, param_stride=(f20 + 3) // 4 * 4, stack_a=P, workspace=None, workspace_bytes=ws),
           dict(frames_b=4, param_stride=(f20 + 3) // 4 * 4, stack_b=P + 4, workspace=P, workspace_bytes=ws)]
    for kw in bad:
        assert L.ss_match_play(ctypes.byref(args(**kw)), None) == -1, kw


def test_match_workspace_grows_with_frames_and_rows():
    from skillshot_learning_b200 import _lib
    W = _lib.lib.ss_match_workspace_bytes
    assert W(1000, 1, 1, 1) == 0 and W(1000, 20, 20, 0) == 0          # no frame-stacked tensor-core forward
    assert W(1000, 20, 1, 1) > W(1000, 1, 1, 1)
    assert W(1000, 1, 4, 1) == W(1000, 4, 4, 1) == W(1000, 20, 4, 1) > 0     # one scratch area, shared by the two forwards
    assert W(100000, 20, 1, 1) > W(1000, 20, 1, 1)
    assert W(0, 1, 1, 1) == -1 and W(10, 0, 1, 1) == -1 and W(10, 1, 21, 1) == -1


def test_match_argument_block_matches_the_header():
    """The ctypes mirror of struct ss_match_args lists the header's fields in the header's order."""
    from skillshot_learning_b200 import _lib
    text = open(os.path.join(ROOT, "include", "skillshot_b200.h")).read()
    body = re.search(r"typedef struct ss_match_args \{(.*?)\} ss_match_args;", text, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = []
    for decl in body.split(";"):
        decl = decl.strip()
        if decl:
            names += [re.sub(r"[\s\*]|const", "", part.split()[-1]) for part in decl.split(",")]
    assert names == [f[0] for f in _lib.MatchArgs._fields_]
    assert _lib.MATCH_STATS == int(re.search(r"#define SS_MATCH_STATS (\d+)", text).group(1))


def test_actor_arguments_are_parsed():
    from skillshot_learning_b200 import _lib
    from skillshot_learning_b200.match import actor_vector
    for f in (1, 4, 20):
        n = int(_lib.lib.ss_actor_frames_params(f))
        v = np.arange(n, dtype=np.float64) * 1e-6
        got, frames = actor_vector(v)
        assert frames == f and got.dtype == np.float32 and np.array_equal(got, v.astype(np.float32))
        shapes = [(12 * f, 256), (256,), (256, 128), (128,), (128, 2), (2,)]
        arrs, o = [], 0
        for sh in shapes:
            k = int(np.prod(sh))
            arrs.append(v[o:o + k].reshape(sh))
            o += k
        got6, frames6 = actor_vector(arrs)
        assert frames6 == f and np.array_equal(got6, got)
    with pytest.raises(ValueError):
        actor_vector(np.zeros(A_N + 1))
    with pytest.raises(ValueError):
        actor_vector(np.zeros((2, A_N)))
    good = [np.zeros(s) for s in [(12, 256), (256,), (256, 128), (128,), (128, 2), (2,)]]
    for bad in ([np.zeros((13, 256))] + good[1:], [np.zeros((252, 256))] + good[1:], good[:5], good[:4] + [np.zeros((128, 3)), good[5]],
                [np.zeros(12 * 256)] + good[1:]):
        with pytest.raises(ValueError):
            actor_vector(bad)


def test_result_arithmetic():
    from skillshot_learning_b200.match import summarize
    c = np.zeros((2, 8), np.int64)
    c[0, :6] = [10, 5, 3, 2, 0, 400]      # A is player 1: 5 wins, 3 losses, 2 draws
    c[1, :6] = [10, 2, 6, 1, 1, 300]
    r = summarize(c)
    assert (r["games"], r["a_wins"], r["b_wins"], r["draws"], r["unfinished"]) == (20, 7, 9, 3, 1)
    assert r["score"] == (7 + 1.5) / 20
    s = np.array([1.0] * 7 + [0.0] * 9 + [0.5] * 3 + [0.0])
    assert math.isclose(r["score_stderr"], s.std(ddof=1) / math.sqrt(20), rel_tol=1e-12)
    assert r["mean_ticks_decided"] == 700 / 16
    p1, p2 = r["by_seat"]["a_player1"], r["by_seat"]["a_player2"]
    assert (p1["games"], p1["a_wins"], p1["b_wins"], p1["draws"], p1["unfinished"]) == (10, 5, 3, 2, 0)
    assert p1["score"] == 0.6 and p1["mean_ticks_decided"] == 50.0
    assert p2["score"] == 0.25 and p2["mean_ticks_decided"] == 300 / 8
    for k in ("games", "a_wins", "b_wins", "draws", "unfinished"):
        assert p1[k] + p2[k] == r[k]
    empty = summarize(np.zeros((2, 8), np.int64))
    assert empty["games"] == 0 and math.isnan(empty["score"]) and math.isnan(empty["mean_ticks_decided"])


# ---------------------------------------------------------------- GPU ------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n", [1000, 65536])
@pytest.mark.parametrize("with_speeds", [False, True])
def test_step_match_equals_env_step_under_the_seat_permutation(n, with_speeds):
    import torch
    from skillshot_learning_b200 import SkillshotEnvs, _lib
    L, st = _lib.lib, torch.cuda.current_stream().cuda_stream
    for split in (0, n // 3, n):
        ref = SkillshotEnvs(n, random_positions=True, seed=7, reward_mode="none", tick_limit=1000, auto_reset=False)
        m = SkillshotEnvs(n, random_positions=True, seed=7, reward_mode="none", tick_limit=1000, auto_reset=False)
        if with_speeds:
            ref.set_speeds(*_speeds(n, 3))
            m.set_speeds(*_speeds(n, 3))
        g = torch.Generator(device="cuda").manual_seed(split + n)
        obs_pm = torch.empty((2, n, 12), device="cuda")
        for t in range(64):
            act_pm = (torch.rand((2, n, 2), device="cuda", generator=g) * 2.4 - 1.2).contiguous()
            out = ref.step(_seat_actions(act_pm, split))
            assert L.ss_env_step_match(m.state.data_ptr(), n, split, act_pm.data_ptr(), obs_pm.data_ptr(), 1000,
                                       None if m.speeds is None else m.speeds.data_ptr(), m.status.data_ptr(), st) == 0
            assert torch.equal(obs_pm, _seat_obs(out["obs"], split)), (split, t)
        assert torch.equal(m.state, ref.state), split
        assert int(m.status.item()) == int(ref.status.item()) == 0


@pytest.mark.gpu
def test_step_match_leaves_a_game_at_the_tick_limit_alone():
    import torch
    from skillshot_learning_b200 import SkillshotEnvs, _lib
    L, st = _lib.lib, torch.cuda.current_stream().cuda_stream
    n, limit = 3000, 8
    m = SkillshotEnvs(n, random_positions=True, seed=1, reward_mode="none", auto_reset=False)
    obs = torch.empty((2, n, 12), device="cuda")
    act = torch.full((2, n, 2), 0.7, device="cuda")
    for _ in range(limit):
        assert L.ss_env_step_match(m.state.data_ptr(), n, n // 2, act.data_ptr(), obs.data_ptr(), limit, None, None, st) == 0
    before, obs_before = m.export_state(), obs.clone()
    live = before["live"] != 0
    assert live.any() and (before["ticks"][live] == limit).all()
    for _ in range(20):
        assert L.ss_env_step_match(m.state.data_ptr(), n, n // 2, act.data_ptr(), obs.data_ptr(), limit, None, None, st) == 0
    after = m.export_state()
    for k in before:
        assert np.array_equal(np.asarray(before[k])[live], np.asarray(after[k])[live]), k
    assert (after["ticks"] <= limit).all()
    assert torch.equal(obs[:, torch.from_numpy(live).cuda()], obs_before[:, torch.from_numpy(live).cuda()])


@pytest.mark.gpu
@pytest.mark.parametrize("groups,rows,short", [(2, 1000, 0), (5, 333, 100), (2, 70001, 3)])
def test_grouped_forward_equals_the_forward_per_group(groups, rows, short):
    import torch
    from skillshot_learning_b200 import _lib
    L, st = _lib.lib, torch.cuda.current_stream().cuda_stream
    n = groups * rows - short                     # the last group is `short` rows shorter
    params = torch.zeros(groups * STRIDE, device="cuda")
    for k in range(groups):
        params[k * STRIDE:k * STRIDE + A_N] = _actor(1, 100 + k).cuda()
    g = torch.Generator(device="cuda").manual_seed(groups)
    obs = torch.rand((n, 12), device="cuda", generator=g)
    act = torch.full((n, 2), float("nan"), device="cuda")
    assert L.ss_actor_forward_groups_tc(params.data_ptr(), STRIDE, rows, obs.data_ptr(), act.data_ptr(), n, st) == 0
    for k in range(groups):
        lo, hi = k * rows, min(n, (k + 1) * rows)
        one = torch.empty((hi - lo, 2), device="cuda")
        sub = obs[lo:hi].contiguous()
        assert L.ss_actor_forward_tc(params[k * STRIDE:].data_ptr(), sub.data_ptr(), one.data_ptr(), hi - lo, 0.0, 1, 0.0, 0, 0, st) == 0
        assert torch.equal(act[lo:hi], one), k


@pytest.mark.gpu
def test_summary_equals_a_host_tally():
    import torch
    from skillshot_learning_b200 import Match
    n, limit = 4096, 150
    m = Match(_actor(1, 1, scale=6.0), _actor(1, 2, scale=6.0), n, tick_limit=limit, seed=3, split=1500)
    for _ in range(3):
        m.advance(40)
        st = m.envs.export_state()
        want = _host_tally(st["ticks"], st["live"], st["winner"], 1500, limit)
        assert np.array_equal(m.counters(), want)
    m.play()
    st = m.envs.export_state()
    c = m.counters()
    assert np.array_equal(c, _host_tally(st["ticks"], st["live"], st["winner"], 1500, limit))
    assert c[:, 4].sum() == 0 and c[:, 1:4].sum() == n and c[:, 1:3].sum() > 0
    torch.cuda.synchronize()


def _stepwise(m, n_ticks):
    """The ticks of ss_match_play composed from the stepwise entry points, on copies of the match's buffers."""
    import torch
    from skillshot_learning_b200 import _lib
    L, st, n = _lib.lib, torch.cuda.current_stream().cuda_stream, m.n_games
    state, obs, act = m.envs.state.clone(), m.obs.clone(), torch.zeros_like(m.act)
    stacks = [None if s is None else s.clone() for s in m.stacks]
    tc = m.precision == "bf16"
    ws = torch.empty(max(16, int(L.ss_actor_frames_tc_workspace_bytes(n, 0))), dtype=torch.uint8, device="cuda")
    head = m.head
    for _ in range(n_ticks):
        for p, f in enumerate((m.frames_a, m.frames_b)):
            prm = m.params[p * m.param_stride:].data_ptr()
            if f > 1 and tc:
                rc = L.ss_actor_forward_frames_tc(prm, 0, 0, stacks[p].data_ptr(), f, head, act[p].data_ptr(), n, ws.data_ptr(), ws.numel(), st)
            elif f > 1:
                rc = L.ss_actor_forward_frames(prm, 0, 0, stacks[p].data_ptr(), f, head, act[p].data_ptr(), n, st)
            elif tc:
                rc = L.ss_actor_forward_tc(prm, obs[p].data_ptr(), act[p].data_ptr(), n, 0.0, 1, 0.0, 0, 0, st)
            else:
                rc = L.ss_actor_forward(prm, obs[p].data_ptr(), act[p].data_ptr(), n, 0.0, 1, 0.0, 0, 0, st)
            assert rc == 0
        assert L.ss_env_step_match(state.data_ptr(), n, m.split, act.data_ptr(), obs.data_ptr(), m.tick_limit,
                                   None, None, st) == 0
        head += 1
        for p, f in enumerate((m.frames_a, m.frames_b)):
            if f > 1:
                push = L.ss_obs_stack_push_tc if tc else L.ss_obs_stack_push
                assert push(stacks[p].data_ptr(), n, f, head, obs[p].data_ptr(), None, 1, st) == 0
    return state, obs, act


@pytest.mark.gpu
@pytest.mark.parametrize("frames", [(1, 1), (20, 1), (4, 4)])
@pytest.mark.parametrize("precision", ["bf16", "f32"])
def test_match_play_equals_the_stepwise_ticks(frames, precision):
    import torch
    from skillshot_learning_b200 import Match
    n = 3000
    m = Match(_actor(frames[0], 11, scale=4.0), _actor(frames[1], 12, scale=4.0), n, precision=precision, tick_limit=500, seed=5,
              split=1100)
    m.advance(3)                               # the same from a history that is not freshly filled
    state, obs, act = _stepwise(m, 37)
    m.advance(37)
    assert torch.equal(m.obs, obs) and torch.equal(m.act, act) and torch.equal(m.envs.state, state)


@pytest.mark.gpu
@pytest.mark.parametrize("random_positions", [False, True])
def test_constant_action_games_equal_the_oracle(random_positions):
    import torch
    from oracle.oracle import OracleEnvs
    from skillshot_learning_b200 import Match
    from tests import philox_ref
    n, limit, split, seed = 2000, 300, 700, 9
    consts = {"a": (0.898, -0.08), "b": (0.189, -0.324)}      # from the fixed start: a hit on player 1 at tick 170 when A is player 1

    def const_actor(c):
        v = torch.zeros(A_N)
        v[-2:] = torch.atanh(torch.tensor(c, dtype=torch.float32))
        return v
    m = Match(const_actor(consts["a"]), const_actor(consts["b"]), n, tick_limit=limit, random_positions=random_positions, seed=seed,
              split=split)
    m.advance(1)
    a_act, b_act = m.act[0, 0].cpu().numpy(), m.act[1, 0].cpu().numpy()     # the float32 actions the kernels produce
    assert (m.act[0] == m.act[0, 0]).all() and (m.act[1] == m.act[1, 0]).all()
    r = m.play()
    orc = OracleEnvs(n, philox_ref.reset_positions(n, seed, 0) if random_positions else None)
    acts = np.empty((n, 2, 2), np.float32)
    acts[:split, 0], acts[:split, 1] = a_act, b_act
    acts[split:, 0], acts[split:, 1] = b_act, a_act
    for _ in range(limit):
        assert orc.step(acts, want_obs=False, reward_mode=0, tick_limit=limit)["errors"] == 0
    want, got = orc.snapshot(), m.envs.export_state()
    assert np.array_equal(got["winner"], want["winner"]) and np.array_equal(got["ticks"], want["ticks"])
    assert np.array_equal(got["live"], want["live"])
    tally = _host_tally(want["ticks"], want["live"], want["winner"], split, limit)
    assert np.array_equal(m.counters(), tally)
    assert r["a_wins"] == tally[:, 1].sum() and r["b_wins"] == tally[:, 2].sum() and r["draws"] == tally[:, 3].sum()
    assert r["a_wins"] + r["b_wins"] > 0 or not random_positions


@pytest.mark.gpu
def test_mirrored_matches_play_the_same_games():
    from skillshot_learning_b200 import Match
    n = 8192
    a, b = _actor(1, 21, scale=6.0), _actor(1, 22, scale=6.0)
    r1 = Match(a, b, n, tick_limit=400, seed=4, split=n).play()
    r2 = Match(b, a, n, tick_limit=400, seed=4, split=0).play()
    assert r1["a_wins"] == r2["b_wins"] and r1["b_wins"] == r2["a_wins"] and r1["draws"] == r2["draws"]
    assert r1["a_wins"] + r1["b_wins"] > 0
    assert r1["by_seat"]["a_player1"]["games"] == n and r2["by_seat"]["a_player2"]["games"] == n


@pytest.mark.gpu
def test_match_is_deterministic_and_respects_the_tick_limit():
    from skillshot_learning_b200 import Match
    args = (_actor(20, 31, scale=5.0), _actor(1, 32, scale=5.0), 5000)
    kw = dict(tick_limit=250, seed=6, split=1234, ticks_per_call=32)
    m1, m2 = Match(*args, **kw), Match(*args, **kw)
    r1, r2 = m1.play(), m2.play()
    assert r1 == r2
    assert r1["unfinished"] == 0 and r1["games"] == 5000
    assert (m1.envs.export_state()["ticks"] <= 250).all()


@pytest.mark.gpu
@pytest.mark.parametrize("frames,precision", [(1, "bf16"), (4, "f32")])
def test_evaluate_does_not_disturb_training(frames, precision):
    import torch
    from skillshot_learning_b200 import ActorCritic, SelfPlayTrainer

    def run(evaluate):
        tr = SelfPlayTrainer(2048, seed=3, batch_size=1024, precision=precision, frames=frames, tick_limit=300)
        res = None
        for k in range(4):
            tr.rollout(4)
            tr.update()
            if evaluate and k == 1:
                res = tr.evaluate(ActorCritic(frames=frames, seed=9).actor, n_games=1024, seed=2, tick_limit=100)
        torch.cuda.synchronize()
        return tr, res
    t1, res = run(True)
    t2, _ = run(False)
    assert res["games"] == 1024 and res["unfinished"] == 0
    assert torch.equal(t1.networks.params, t2.networks.params) and torch.equal(t1.networks.target, t2.networks.target)
    assert torch.equal(t1.envs.state, t2.envs.state) and torch.equal(t1.replay.obs, t2.replay.obs)
    assert t1.envs.counter == t2.envs.counter and t1.networks.counter == t2.networks.counter
