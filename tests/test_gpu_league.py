"""Leagues of many actors (ss_env_step_seated, ss_actor_forward_segments_tc, ss_league_summary, ss_league_play, League,
ratings, load_saved_actors, SelfPlayTrainer.evaluate_league).  The GPU tests compare with ==: the seated step against
ss_env_step and ss_env_step_match, the segment forward against ss_actor_forward_tc per segment and the grouped forward,
the summary against a host tally, the one-call league against its stepwise composition, and a two-policy league against
Match.  The unmarked tests run without a GPU: argument rejection, the argument block's field order, the schedules, the
checkpoint loader and the rating fit."""
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
def _actor(frames, seed, scale=1.0):
    import torch
    from skillshot_learning_b200 import _lib
    n = int(_lib.lib.ss_actor_frames_params(frames))
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(n, generator=g) * 0.05 * scale).float()


def _speeds(n, seed):
    rng = np.random.default_rng(seed)
    return (rng.uniform(1.0, 5.0, n), rng.uniform(0.05, 0.5, n), rng.uniform(2.0, 8.0, n), rng.integers(5, 30, n))


def _league_tally(ticks, live, winner, seat_policy, P, tick_limit):
    """[P][P][8] counters of ss_league_summary from exported state (winner_id = the player HIT)."""
    out = np.zeros((P, P, 8), np.int64)
    for e in range(ticks.size):
        c = out[seat_policy[e, 0], seat_policy[e, 1]]
        c[0] += 1
        if not live[e]:
            c[1 if winner[e] == 2 else 2] += 1
            c[5] += ticks[e]
        else:
            c[3 if ticks[e] >= tick_limit else 4] += 1
    return out


def _args(P=3, n=96, **kw):
    from skillshot_learning_b200 import _lib
    Q = 4096
    a = _lib.LeagueArgs()
    seg = (ctypes.c_int64 * (P + 1))(*[2 * n * s // P for s in range(P + 1)])
    fr = (ctypes.c_int * P)(*([1] * P))
    st = (ctypes.c_void_p * P)(*([Q] * P))
    a.state, a.n_envs, a.tick_limit, a.seat_rows, a.obs, a.act, a.params, a.param_stride = Q, n, 50, Q, Q, Q, Q, STRIDE
    a.n_policies, a.head, a.tensor_cores, a.n_ticks = P, 0, 1, 4
    a.seg_start = ctypes.cast(seg, ctypes.POINTER(ctypes.c_int64))
    a.frames = ctypes.cast(fr, ctypes.POINTER(ctypes.c_int))
    a.stacks = ctypes.cast(st, ctypes.POINTER(ctypes.c_void_p))
    a._keep = (seg, fr, st)
    for k, v in kw.items():
        setattr(a, k, v)
    return a, seg, fr, st


# ---------------------------------------------------------------- CPU ------------------------------------------------------------------
def test_league_entry_points_reject_bad_arguments_without_a_gpu():
    from skillshot_learning_b200 import _lib
    L = _lib.lib
    P, Q = 4096, 4097
    assert L.ss_env_step_seated(None, 16, P, 32, P, P, 100, None, None, None) == -1
    assert L.ss_env_step_seated(P, 16, None, 32, P, P, 100, None, None, None) == -1
    assert L.ss_env_step_seated(P, 16, P, 0, P, P, 100, None, None, None) == -1
    assert L.ss_env_step_seated(P, 16, P, 1 << 31, P, P, 100, None, None, None) == -1
    assert L.ss_env_step_seated(P, 16, P, 32, P, P, 0, None, None, None) == -1
    assert L.ss_env_step_seated(Q, 16, P, 32, P, P, 100, None, None, None) == -1
    assert L.ss_env_step_seated(P, 16, P + 4, 32, P, P, 100, None, None, None) == -1
    assert L.ss_env_step_seated(P, 16, P, 32, P + 4, P, 100, None, None, None) == -1
    assert L.ss_env_step_seated(P, 16, P, 32, P, P + 8, 100, None, None, None) == -1
    rows = (ctypes.c_int64 * 65)(*([100] * 65))
    assert L.ss_actor_forward_segments_tc(None, STRIDE, rows, 2, P, P, None) == -1
    assert L.ss_actor_forward_segments_tc(P, STRIDE, None, 2, P, P, None) == -1
    assert L.ss_actor_forward_segments_tc(P, STRIDE, rows, 0, P, P, None) == -1
    assert L.ss_actor_forward_segments_tc(P, STRIDE, rows, 65, P, P, None) == -1          # more than 64 segments
    assert L.ss_actor_forward_segments_tc(P, STRIDE + 2, rows, 2, P, P, None) == -1
    assert L.ss_actor_forward_segments_tc(P, 1024, rows, 2, P, P, None) == -1
    assert L.ss_actor_forward_segments_tc(P + 4, STRIDE, rows, 2, P, P, None) == -1
    assert L.ss_actor_forward_segments_tc(P, STRIDE, rows, 2, P, P + 4, None) == -1
    empty = (ctypes.c_int64 * 2)(100, 0)
    assert L.ss_actor_forward_segments_tc(P, STRIDE, empty, 2, P, P, None) == -1          # an empty segment
    assert L.ss_league_summary(None, 16, P, 3, 100, P, None) == -1
    assert L.ss_league_summary(P, 16, None, 3, 100, P, None) == -1
    assert L.ss_league_summary(P, 16, P, 1, 100, P, None) == -1
    assert L.ss_league_summary(P, 16, P, 65, 100, P, None) == -1                             # P > 64
    assert L.ss_league_summary(P, 16, P, 3, 0, P, None) == -1
    assert L.ss_league_summary(P, 16, P + 1, 3, 100, P, None) == -1
    assert L.ss_league_summary(P, 16, P, 3, 100, P + 4, None) == -1
    assert L.ss_league_play(None, None) == -1 and L.ss_league_workspace_bytes(None) == -1

    good, _, _, _ = _args()
    assert L.ss_league_workspace_bytes(ctypes.byref(good)) == 0
    f20 = (int(L.ss_actor_frames_params(20)) + 3) // 4 * 4
    bad = [dict(state=None), dict(obs=None), dict(act=None), dict(params=None), dict(seat_rows=None), dict(state=Q),
           dict(obs=P + 8), dict(act=P + 4), dict(params=P + 4), dict(seat_rows=P + 4), dict(speeds=P + 8), dict(status=P + 2),
           dict(n_envs=0), dict(n_envs=97), dict(tick_limit=0), dict(n_ticks=0), dict(head=-1), dict(param_stride=STRIDE - 4),
           dict(param_stride=STRIDE + 2), dict(n_policies=1), dict(n_policies=65)]
    for kw in bad:
        a, _, _, _ = _args(**kw)
        assert L.ss_league_play(ctypes.byref(a), None) == -1, kw
    # segments: not starting at 0, not increasing (non-contiguous), an empty one, not summing to 2 n_envs
    for seg in ([1, 64, 128, 192], [0, 100, 64, 192], [0, 64, 64, 192], [0, 64, 128, 190]):
        a, s, _, _ = _args()
        for k, v in enumerate(seg):
            s[k] = v
        assert L.ss_league_play(ctypes.byref(a), None) == -1, seg
    a, _, fr, _ = _args()
    fr[1] = 21
    assert L.ss_league_play(ctypes.byref(a), None) == -1 and L.ss_league_workspace_bytes(ctypes.byref(a)) == -1
    # a 20-frame segment: its history, the stride and the workspace
    a, _, fr, st = _args(param_stride=f20)
    fr[2] = 20
    ws = int(L.ss_league_workspace_bytes(ctypes.byref(a)))
    assert ws > 0
    a.workspace, a.workspace_bytes = P, ws - 1
    assert L.ss_league_play(ctypes.byref(a), None) == -1                                     # short workspace
    a.workspace, a.workspace_bytes = None, ws
    assert L.ss_league_play(ctypes.byref(a), None) == -1
    a.workspace, a.workspace_bytes, a.param_stride = P, ws, STRIDE
    assert L.ss_league_play(ctypes.byref(a), None) == -1                                     # stride shorter than the vector
    a.param_stride = f20
    st[2] = None
    assert L.ss_league_play(ctypes.byref(a), None) == -1                                     # no history
    st[2] = P + 4
    assert L.ss_league_play(ctypes.byref(a), None) == -1
    a.tensor_cores = 0
    assert L.ss_league_workspace_bytes(ctypes.byref(a)) == 0


def test_league_argument_block_matches_the_header():
    """The ctypes mirror of struct ss_league_args lists the header's fields in the header's order."""
    from skillshot_learning_b200 import _lib
    text = open(os.path.join(ROOT, "include", "skillshot_b200.h")).read()
    body = re.search(r"typedef struct ss_league_args \{(.*?)\} ss_league_args;", text, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = []
    for decl in body.split(";"):
        decl = decl.strip()
        if decl:
            names += [re.sub(r"[\s\*]|const", "", part.split()[-1]) for part in decl.split(",")]
    assert names == [f[0] for f in _lib.LeagueArgs._fields_]
    assert _lib.LEAGUE_MAX_POLICIES == int(re.search(r"#define SS_LEAGUE_MAX_POLICIES (\d+)", text).group(1))
    assert _lib.STATUS_SEAT_RANGE == int(re.search(r"#define SS_STATUS_SEAT_RANGE (\d+)", text).group(1))


def test_schedules_are_complete_and_seat_balanced():
    from skillshot_learning_b200.league import gauntlet, round_robin
    for P in (2, 5, 64):
        rr = round_robin(P)
        assert len(rr) == P * (P - 1) // 2 and len({frozenset(p) for p in rr}) == len(rr) and all(i != j for i, j in rr)
        assert gauntlet(P) == [(0, j) for j in range(1, P)]
    # the env layout of a league: every pair plays g / 2 games in each seat order
    g, pairs = 6, round_robin(4)
    pol = np.empty((len(pairs) * g, 2), np.int64)
    for k, (i, j) in enumerate(pairs):
        pol[k * g:k * g + g // 2] = (i, j)
        pol[k * g + g // 2:(k + 1) * g] = (j, i)
    for i, j in pairs:
        assert ((pol[:, 0] == i) & (pol[:, 1] == j)).sum() == ((pol[:, 0] == j) & (pol[:, 1] == i)).sum() == g // 2


def test_load_saved_actors_reads_checkpoints_in_epoch_order(tmp_path):
    from skillshot_learning_b200.league import load_saved_actors
    from skillshot_learning_b200.match import actor_vector
    d = tmp_path / "actor"
    d.mkdir()
    shapes = [(12, 256), (256,), (256, 128), (128,), (128, 2), (2,)]
    for start, end in ((0, 100), (100, 1000), (1000, 20), (20, 200)):
        np.savez(d / ("%d_%d_model.npz" % (start, end)), *[np.full(s, end, np.float32) for s in shapes])
    (d / "notes.txt").write_text("not a model")
    got = load_saved_actors(str(tmp_path))
    assert [n for n, _ in got] == ["1000_20", "0_100", "20_200", "100_1000"]
    for name, arrs in got:
        assert [a.shape for a in arrs] == shapes and float(arrs[0][0, 0]) == float(name.split("_")[1])
        assert actor_vector(arrs)[1] == 1
    assert load_saved_actors(str(tmp_path / "missing")) == []


def _counts(P, pairs, wins_ij, draws_ij, games):
    """[P][P][8] counters with games / 2 per seat order; wins_ij[k], draws_ij[k]: pair k's wins of i and draws, split
    evenly over the seats."""
    c = np.zeros((P, P, 8), np.int64)
    for k, (i, j) in enumerate(pairs):
        w, d = int(wins_ij[k]), int(draws_ij[k])
        lo = games - w - d
        for (a, b), ww, ll, dd in (((i, j), w // 2, lo // 2, d // 2), ((j, i), lo - lo // 2, w - w // 2, d - d // 2)):
            c[a, b, 0] = ww + ll + dd
            c[a, b, 1], c[a, b, 2], c[a, b, 3] = ww, ll, dd
    return c


def test_ratings_of_two_policies_are_the_logit_of_the_score():
    from skillshot_learning_b200.league import ratings
    for w, d, g in ((70, 10, 100), (100, 0, 100), (0, 0, 40), (13, 30, 60)):
        c = _counts(2, [(0, 1)], [w], [d], g)
        r, se = ratings(c)
        s = (w + d / 2 + 0.5) / (g + 1)               # after the virtual draw
        assert math.isclose(r[0] - r[1], 400 * math.log10(s / (1 - s)), rel_tol=1e-9, abs_tol=1e-9)
        assert math.isclose(r[0] + r[1], 0.0, abs_tol=1e-9)
        # the inverse Fisher information of one pair: var(theta_0 - theta_1) = 1 / (n s (1 - s)), split over two anchored ratings
        want = 400 / math.log(10) * 0.5 / math.sqrt((g + 1) * s * (1 - s))
        assert math.isclose(se[0], want, rel_tol=1e-6) and math.isclose(se[1], want, rel_tol=1e-6)


def test_ratings_recover_known_strengths():
    from skillshot_learning_b200.league import ratings, round_robin
    rng = np.random.default_rng(5)
    P, g = 8, 4000
    true = rng.normal(0, 1.0, P)
    true -= true.mean()
    pairs = round_robin(P)
    p = [1 / (1 + math.exp(true[j] - true[i])) for i, j in pairs]
    wins = [rng.binomial(g, q) for q in p]
    r, se = ratings(_counts(P, pairs, wins, [0] * len(pairs), g))
    elo = true * 400 / math.log(10)
    assert np.all(np.abs(r - elo) < 3 * se), (r - elo) / se
    assert abs(r.sum()) < 1e-6 and np.all(se > 0)


def test_ratings_follow_a_permutation_and_reject_a_disconnected_schedule():
    from skillshot_learning_b200.league import gauntlet, ratings, round_robin
    rng = np.random.default_rng(2)
    P = 6
    pairs = round_robin(P)
    c = _counts(P, pairs, rng.integers(0, 60, len(pairs)), rng.integers(0, 20, len(pairs)), 80)
    r, se = ratings(c)
    perm = rng.permutation(P)
    cp = c[np.ix_(perm, perm)]
    rp, sep = ratings(cp)
    assert np.allclose(rp, r[perm], atol=1e-8) and np.allclose(sep, se[perm], atol=1e-8)
    g = _counts(P, gauntlet(P), [30] * (P - 1), [5] * (P - 1), 60)
    assert np.isfinite(ratings(g)[0]).all()
    split = _counts(4, [(0, 1), (2, 3)], [10, 10], [0, 0], 20)
    with pytest.raises(ValueError):
        ratings(split)


# ---------------------------------------------------------------- GPU ------------------------------------------------------------------
def _random_seating(n, rng):
    """a random seat table: rows a permutation of [0, 2 n)"""
    perm = rng.permutation(2 * n).astype(np.int32)
    return perm.reshape(n, 2)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1000, 65536])
@pytest.mark.parametrize("with_speeds", [False, True])
def test_seated_step_equals_env_step_under_the_seat_permutation(n, with_speeds):
    import torch
    from skillshot_learning_b200 import SkillshotEnvs, _lib
    L, st = _lib.lib, torch.cuda.current_stream().cuda_stream
    rng = np.random.default_rng(n + with_speeds)
    rows_h = _random_seating(n, rng)
    rows = torch.from_numpy(rows_h).cuda()
    rl = rows.long()
    ref = SkillshotEnvs(n, random_positions=True, seed=7, reward_mode="none", tick_limit=1000, auto_reset=False)
    m = SkillshotEnvs(n, random_positions=True, seed=7, reward_mode="none", tick_limit=1000, auto_reset=False)
    if with_speeds:
        ref.set_speeds(*_speeds(n, 3))
        m.set_speeds(*_speeds(n, 3))
    g = torch.Generator(device="cuda").manual_seed(n)
    obs = torch.empty((2 * n, 12), device="cuda")
    for t in range(48):
        act = (torch.rand((2 * n, 2), device="cuda", generator=g) * 2.4 - 1.2).contiguous()
        out = ref.step(torch.stack([act[rl[:, 0]], act[rl[:, 1]]], dim=1).contiguous())
        assert L.ss_env_step_seated(m.state.data_ptr(), n, rows.data_ptr(), 2 * n, act.data_ptr(), obs.data_ptr(), 1000,
                                    None if m.speeds is None else m.speeds.data_ptr(), m.status.data_ptr(), st) == 0
        assert torch.equal(obs[rl[:, 0]], out["obs"][:, 0]) and torch.equal(obs[rl[:, 1]], out["obs"][:, 1]), t
    assert torch.equal(m.state, ref.state)
    assert int(m.status.item()) == int(ref.status.item()) == 0


@pytest.mark.gpu
def test_seated_step_with_the_split_table_equals_the_match_step_and_guards_its_rows():
    import torch
    from skillshot_learning_b200 import SkillshotEnvs, _lib
    L, st = _lib.lib, torch.cuda.current_stream().cuda_stream
    n, split = 5000, 1700
    i = np.arange(n)
    rows_h = np.stack([np.where(i < split, i, n + i), np.where(i < split, n + i, i)], 1).astype(np.int32)
    rows = torch.from_numpy(rows_h).cuda()
    a = SkillshotEnvs(n, random_positions=True, seed=2, reward_mode="none", auto_reset=False)
    b = SkillshotEnvs(n, random_positions=True, seed=2, reward_mode="none", auto_reset=False)
    oa, ob = torch.empty((2 * n, 12), device="cuda"), torch.empty((2 * n, 12), device="cuda")
    g = torch.Generator(device="cuda").manual_seed(1)
    for _ in range(40):
        act = (torch.rand((2 * n, 2), device="cuda", generator=g) * 2.4 - 1.2).contiguous()
        assert L.ss_env_step_match(a.state.data_ptr(), n, split, act.data_ptr(), oa.data_ptr(), 30, None, a.status.data_ptr(), st) == 0
        assert L.ss_env_step_seated(b.state.data_ptr(), n, rows.data_ptr(), 2 * n, act.data_ptr(), ob.data_ptr(), 30, None,
                                    b.status.data_ptr(), st) == 0
    assert torch.equal(oa, ob) and torch.equal(a.state, b.state) and int(b.status.item()) == 0
    # rows outside [0, n_rows): those envs are not stepped, their rows not written, and the status says so
    bad = rows_h.copy()
    bad[10, 0], bad[20, 1], bad[30, 0] = -1, 2 * n, 1 << 30
    badt = torch.from_numpy(bad).cuda()
    before = b.export_state()
    out = torch.full_like(ob, float("nan"))
    act = torch.zeros((2 * n, 2), device="cuda")
    assert L.ss_env_step_seated(b.state.data_ptr(), n, badt.data_ptr(), 2 * n, act.data_ptr(), out.data_ptr(), 1000, None,
                                b.status.data_ptr(), st) == 0
    assert int(b.status.item()) == _lib.STATUS_SEAT_RANGE
    after, skip = b.export_state(), [10, 20, 30]
    for k in before:
        assert np.array_equal(np.asarray(before[k])[skip], np.asarray(after[k])[skip]), k
    written = torch.ones(2 * n, dtype=torch.bool, device="cuda")
    written[torch.from_numpy(rows_h[skip].ravel().astype(np.int64)).cuda()] = False
    assert torch.isnan(out[~written]).all() and not torch.isnan(out[written]).any()


def _seg_params(k, frames=1):
    import torch
    params = torch.zeros(k * STRIDE, device="cuda")
    for s in range(k):
        params[s * STRIDE:s * STRIDE + A_N] = _actor(frames, 300 + s).cuda()
    return params


@pytest.mark.gpu
@pytest.mark.parametrize("lengths", [[1, 127, 128, 129], [70001, 1, 300], [129] * 3 + [128 * 40], "64"])
def test_segment_forward_equals_the_forward_per_segment(lengths):
    import torch
    from skillshot_learning_b200 import _lib
    L, st = _lib.lib, torch.cuda.current_stream().cuda_stream
    if lengths == "64":
        lengths = list(np.random.default_rng(0).integers(1, 900, 64))
    k, n = len(lengths), int(sum(lengths))
    params = _seg_params(k)
    g = torch.Generator(device="cuda").manual_seed(k)
    obs = torch.rand((n, 12), device="cuda", generator=g)
    act = torch.full((n, 2), float("nan"), device="cuda")
    rows = (ctypes.c_int64 * k)(*[int(v) for v in lengths])
    assert L.ss_actor_forward_segments_tc(params.data_ptr(), STRIDE, rows, k, obs.data_ptr(), act.data_ptr(), st) == 0
    lo = 0
    for s, m in enumerate(lengths):
        m = int(m)
        one = torch.empty((m, 2), device="cuda")
        sub = obs[lo:lo + m].contiguous()
        assert L.ss_actor_forward_tc(params[s * STRIDE:].data_ptr(), sub.data_ptr(), one.data_ptr(), m, 0.0, 1, 0.0, 0, 0, st) == 0
        assert torch.equal(act[lo:lo + m], one), s
        lo += m


@pytest.mark.gpu
def test_uniform_segments_equal_the_grouped_forward():
    import torch
    from skillshot_learning_b200 import _lib
    L, st = _lib.lib, torch.cuda.current_stream().cuda_stream
    k, m = 16, 4096
    params = _seg_params(k)
    obs = torch.rand((k * m, 12), device="cuda", generator=torch.Generator(device="cuda").manual_seed(3))
    a1, a2 = torch.empty((k * m, 2), device="cuda"), torch.empty((k * m, 2), device="cuda")
    rows = (ctypes.c_int64 * k)(*([m] * k))
    assert L.ss_actor_forward_segments_tc(params.data_ptr(), STRIDE, rows, k, obs.data_ptr(), a1.data_ptr(), st) == 0
    assert L.ss_actor_forward_groups_tc(params.data_ptr(), STRIDE, m, obs.data_ptr(), a2.data_ptr(), k * m, st) == 0
    assert torch.equal(a1, a2)


@pytest.mark.gpu
@pytest.mark.parametrize("P", [2, 5, 64])
def test_league_summary_equals_a_host_tally(P):
    from skillshot_learning_b200 import League
    from skillshot_learning_b200.league import round_robin
    pairs = round_robin(P) if P < 64 else [(i, (i + 1) % P) for i in range(P)] + [(i, (i + 7) % P) for i in range(P)]
    g = 64 if P < 64 else 32
    lg = League([_actor(1, 40 + p, scale=6.0) for p in range(P)], g, pairs=pairs, tick_limit=120, seed=3)
    for _ in range(2):
        lg.advance(50)
        s = lg.envs.export_state()
        want = _league_tally(s["ticks"], s["live"], s["winner"], lg.seat_policy_host, P, 120)
        assert np.array_equal(lg.counters(), want)
    r = lg.play()
    s = lg.envs.export_state()
    c = lg.counters()
    assert np.array_equal(c, _league_tally(s["ticks"], s["live"], s["winner"], lg.seat_policy_host, P, 120))
    assert r["unfinished"] == 0 and r["games"] == len(pairs) * g and c[:, :, 1:3].sum() > 0


def _stepwise(lg, n_ticks):
    """The ticks of ss_league_play composed from the stepwise entry points, on copies of the league's buffers."""
    import torch
    from skillshot_learning_b200 import _lib
    L, st, n = _lib.lib, torch.cuda.current_stream().cuda_stream, lg.n_envs
    state, obs, act = lg.envs.state.clone(), lg.obs.clone(), torch.zeros_like(lg.act)
    stacks = [None if s is None else s.clone() for s in lg.stacks]
    tc = lg.precision == "bf16"
    ws = torch.empty(max(16, int(L.ss_actor_frames_tc_workspace_bytes(2 * n, 0))), dtype=torch.uint8, device="cuda")
    head = lg.head
    seg = lg.seg_start
    for _ in range(n_ticks):
        for s, p in enumerate(lg.order):
            f, lo, m = lg.frames[p], int(seg[s]), int(seg[s + 1] - seg[s])
            prm = lg.params[s * lg.param_stride:].data_ptr()
            a, o = act[lo:].data_ptr(), obs[lo:].data_ptr()
            if f > 1 and tc:
                rc = L.ss_actor_forward_frames_tc(prm, 0, 0, stacks[s].data_ptr(), f, head, a, m, ws.data_ptr(), ws.numel(), st)
            elif f > 1:
                rc = L.ss_actor_forward_frames(prm, 0, 0, stacks[s].data_ptr(), f, head, a, m, st)
            elif tc:
                rc = L.ss_actor_forward_tc(prm, o, a, m, 0.0, 1, 0.0, 0, 0, st)
            else:
                rc = L.ss_actor_forward(prm, o, a, m, 0.0, 1, 0.0, 0, 0, st)
            assert rc == 0
        assert L.ss_env_step_seated(state.data_ptr(), n, lg.seat_rows.data_ptr(), 2 * n, act.data_ptr(), obs.data_ptr(),
                                    lg.tick_limit, None, None, st) == 0
        head += 1
        for s, p in enumerate(lg.order):
            f, lo, m = lg.frames[p], int(seg[s]), int(seg[s + 1] - seg[s])
            if f > 1:
                push = L.ss_obs_stack_push_tc if tc else L.ss_obs_stack_push
                assert push(stacks[s].data_ptr(), m, f, head, obs[lo:].data_ptr(), None, 1, st) == 0
    return state, obs, act


@pytest.mark.gpu
@pytest.mark.parametrize("frames", [(1, 1, 1), (1, 20, 4), (4, 4)])
@pytest.mark.parametrize("precision", ["bf16", "f32"])
def test_league_play_equals_the_stepwise_ticks(frames, precision):
    import torch
    from skillshot_learning_b200 import League
    actors = [_actor(f, 60 + k, scale=4.0) for k, f in enumerate(frames)]
    lg = League(actors, 1000, precision=precision, tick_limit=500, seed=5)
    lg.advance(3)
    state, obs, act = _stepwise(lg, 29)
    lg.advance(29)
    assert torch.equal(lg.obs, obs) and torch.equal(lg.act, act) and torch.equal(lg.envs.state, state)


@pytest.mark.gpu
@pytest.mark.parametrize("frames", [(1, 1), (20, 1)])
def test_two_policy_league_is_a_match(frames):
    from skillshot_learning_b200 import League, Match
    g = 6000
    a, b = _actor(frames[0], 81, scale=6.0), _actor(frames[1], 82, scale=6.0)
    lg = League([a, b], g, tick_limit=300, seed=4)
    r = lg.play()
    m = Match(a, b, g, tick_limit=300, seed=4, split=g // 2)
    m.play()
    cm, cl = m.counters(), lg.counters()
    assert np.array_equal(cl[0, 1], cm[0]) and np.array_equal(cl[1, 0, :6], cm[1, [0, 2, 1, 3, 4, 5]])
    assert cl[0, 0, 0] == cl[1, 1, 0] == 0
    assert (lg.envs.export_state()["ticks"] <= 300).all() and r["unfinished"] == 0
    # swapping the actors (with the pair written the other way round, so that the same envs seat the same actor first)
    # mirrors the table
    c2 = League([b, a], g, pairs=[(1, 0)], tick_limit=300, seed=4)
    r2 = c2.play()
    c2 = c2.counters()
    assert np.array_equal(c2[1, 0], cl[0, 1]) and np.array_equal(c2[0, 1], cl[1, 0])
    assert np.allclose(r2["ratings"], r["ratings"][::-1]) and r2["policies"][1] == r["policies"][0]
    # two runs give identical results
    r3 = League([a, b], g, tick_limit=300, seed=4).play()
    assert r3["pairs"] == r["pairs"] and np.array_equal(r3["ratings"], r["ratings"])


@pytest.mark.gpu
@pytest.mark.parametrize("frames,precision", [(1, "bf16"), (4, "f32")])
def test_evaluate_league_does_not_disturb_training(frames, precision):
    import torch
    from skillshot_learning_b200 import ActorCritic, SelfPlayTrainer

    def run(evaluate):
        tr = SelfPlayTrainer(2048, seed=3, batch_size=1024, precision=precision, frames=frames, tick_limit=300)
        res = None
        for k in range(4):
            tr.rollout(4)
            tr.update()
            if evaluate and k == 1:
                res = tr.evaluate_league([ActorCritic(frames=frames, seed=9 + s).actor for s in range(3)], games_per_pair=512,
                                         seed=2, tick_limit=100)
        torch.cuda.synchronize()
        return tr, res
    t1, res = run(True)
    t2, _ = run(False)
    assert res["games"] == 3 * 512 and res["unfinished"] == 0 and len(res["ratings"]) == 4
    assert np.isnan(res["score"][1, 2]) and not np.isnan(res["score"][0, 2])
    assert torch.equal(t1.networks.params, t2.networks.params) and torch.equal(t1.networks.target, t2.networks.target)
    assert torch.equal(t1.envs.state, t2.envs.state) and torch.equal(t1.replay.obs, t2.replay.obs)
    assert t1.envs.counter == t2.envs.counter and t1.networks.counter == t2.networks.counter
