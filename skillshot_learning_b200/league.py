"""Leagues: many actors playing a schedule of pairings in one batch on one GPU, and their Bradley-Terry ratings
(ss_league_play, include/skillshot_b200.h).

A :class:`Match` answers "does A beat B".  A training run asks that of many checkpoints at once, and pairwise scores cannot
be combined into one ordering: they are not transitive and some pairs are never played.  A :class:`League` plays every
scheduled pair (a round robin, a gauntlet of one candidate against a pool, or any list of pairs) in one batch of envs and
fits one rating per policy, with standard errors, to all the games.

Layout (the contract of the kernels):

* envs are pair-major: pair k = (i, j) of the schedule owns envs [k g, (k + 1) g), g = games_per_pair; policy i is player 1
  in the first g / 2 of them and policy j in the last g / 2.  With two policies and the schedule [(0, 1)] a league plays
  exactly the games of ``Match(a0, a1, g, split=g // 2)`` with the same seed (the random starts are keyed by env index);
* the observation and action rows are policy-major: one segment per policy, one row for every env in which it plays, in
  env order; the 1-frame policies' segments come first so that their forwards are one launch;
* ``winner_id`` is the id of the player that was HIT, as in a match.
"""
from __future__ import annotations

import ctypes
import glob
import math
import os

import numpy as np
import torch

from . import _lib
from ._lib import check, lib
from .game import SkillshotEnvs
from .match import _block, _stream, actor_vector

ELO = 400.0 / math.log(10.0)          # rating points per unit of log-strength


def round_robin(n_policies: int) -> list:
    """Every unordered pair (i, j), i < j, of n_policies policies."""
    return [(i, j) for i in range(n_policies) for j in range(i + 1, n_policies)]


def gauntlet(n_policies: int) -> list:
    """Policy 0 against each of the others: (0, j) for j = 1 .. n_policies - 1."""
    return [(0, j) for j in range(1, n_policies)]


def _components(n: int, edges) -> int:
    parent = list(range(n))

    def find(x):
        while parent[x] != x:
            parent[x] = parent[parent[x]]
            x = parent[x]
        return x
    for i, j in edges:
        parent[find(i)] = find(j)
    return len({find(x) for x in range(n)})


def ratings(counters, tol: float = 1e-10, max_iter: int = 100):
    """Bradley-Terry ratings (Elo scale) and their standard errors from league counters [P][P][8] (ss_league_summary:
    cell (i, j) = games with i in seat 1 and j in seat 2, then seat-1 wins, seat-2 wins, draws, ...).

    Model: P(i beats j) = 1 / (1 + exp(theta_j - theta_i)).  A draw counts as half a win for each side, unfinished games
    are left out, and ONE VIRTUAL DRAW is added to every scheduled pair (every pair with a game in either seat order), so
    that a clean sweep still has a finite maximum.  The likelihood is maximised by Newton's method with step halving until
    the largest step is below `tol` (in units of log-strength).  Ratings are 400 / ln 10 rating points per unit of
    log-strength, anchored so that they sum to 0; the standard errors are the square roots of the diagonal of the inverse
    Fisher information of that anchored problem (the pseudo-inverse of the information matrix, whose null space is the
    common shift).  Returns (ratings, stderr), float64 arrays of P.  Raises ValueError when the scheduled pairs do not
    connect all policies: their ratings would not be comparable."""
    c = np.asarray(counters, dtype=np.float64)
    if c.ndim != 3 or c.shape[0] != c.shape[1] or c.shape[2] < 4:
        raise ValueError("counters must be [P][P][8], got shape %s" % (c.shape,))
    P = c.shape[0]
    # wins[i, j]: i's score against j over both seat orders (seat-1 wins of cell (i, j), seat-2 wins of cell (j, i))
    wins = c[:, :, 1] + c[:, :, 2].T + (c[:, :, 3] + c[:, :, 3].T) / 2
    games = c[:, :, 1] + c[:, :, 2] + c[:, :, 3]
    games = games + games.T
    played = (c[:, :, 0] + c[:, :, 0].T) > 0
    np.fill_diagonal(played, False)
    wins = wins + 0.5 * played
    games = games + played
    if _components(P, zip(*np.nonzero(np.triu(played)))) != 1:
        raise ValueError("the scheduled pairs do not connect all %d policies: their ratings are not comparable" % P)

    def loglik(th):
        d = th[:, None] - th[None, :]
        # sum over i < j of w_ij log s(d_ij) + w_ji log s(-d_ij) = w_ij d_ij - n_ij log(1 + e^d_ij)
        return float(np.sum(np.triu(wins * d - games * np.logaddexp(0.0, d), 1)))

    def info(th):
        p = 1.0 / (1.0 + np.exp(-(th[:, None] - th[None, :])))
        w = games * p * (1 - p)
        return np.diag(w.sum(1)) - w, p

    ones = np.full((P, P), 1.0 / P)
    th = np.zeros(P)
    for _ in range(max_iter):
        L, p = info(th)
        grad = (wins - games * p).sum(1)
        step = np.linalg.solve(L + ones, grad)           # = L^+ grad: the sum-zero Newton step (grad sums to 0)
        step -= step.mean()
        f0, t = loglik(th), 1.0
        while loglik(th + t * step) < f0 - 1e-12 and t > 1e-8:
            t /= 2
        th = th + t * step
        if np.max(np.abs(t * step)) < tol:
            break
    else:
        raise RuntimeError("the Bradley-Terry fit did not converge in %d iterations" % max_iter)
    th -= th.mean()
    L, _ = info(th)
    cov = np.linalg.inv(L + ones) - ones                  # Moore-Penrose inverse of the Laplacian-shaped information
    return ELO * th, ELO * np.sqrt(np.maximum(np.diag(cov), 0.0))


def _score(wins, draws, games):
    """(score, stderr) of per-game scores 1 / 0.5 / 0 (the sample variance, as match.summarize)."""
    if games == 0:
        return float("nan"), float("nan")
    mean = (wins + draws / 2) / games
    if games < 2:
        return mean, float("nan")
    var = ((wins + draws / 4) - games * mean * mean) / (games - 1)
    return mean, math.sqrt(max(var, 0.0) / games)


def summarize(counters, pairs) -> dict:
    """The result dict of League.play from int [P][P][8] counters and the schedule (see League.play)."""
    c = np.asarray(counters, dtype=np.int64)
    P = c.shape[0]
    score = np.full((P, P), np.nan)
    score_se = np.full((P, P), np.nan)
    out_pairs, by_seat = [], {}
    for i, j in pairs:
        g = c[i, j] + c[j, i]
        i_wins, j_wins = int(c[i, j, 1] + c[j, i, 2]), int(c[i, j, 2] + c[j, i, 1])
        draws = int(g[3])
        s, se = _score(i_wins, draws, int(i_wins + j_wins + draws))
        score[i, j], score_se[i, j] = s, se
        score[j, i], score_se[j, i] = 1 - s, se
        out_pairs.append(dict(pair=(i, j), games=int(g[0]), i_wins=i_wins, j_wins=j_wins, draws=draws, unfinished=int(g[4]),
                              score=s, score_stderr=se))
        for a, b in ((i, j), (j, i)):
            blk = _block(c[a, b])
            by_seat[(a, b)] = dict(games=blk["games"], seat1_wins=blk["a_wins"], seat2_wins=blk["b_wins"], draws=blk["draws"],
                                   unfinished=blk["unfinished"], seat1_score=blk["score"],
                                   mean_ticks_decided=blk["mean_ticks_decided"])
    policies = []
    for p in range(P):
        w = int(c[p, :, 1].sum() + c[:, p, 2].sum())
        lo = int(c[p, :, 2].sum() + c[:, p, 1].sum())
        d = int(c[p, :, 3].sum() + c[:, p, 3].sum())
        u = int(c[p, :, 4].sum() + c[:, p, 4].sum())
        s, se = _score(w, d, w + lo + d)
        policies.append(dict(games=int(c[p, :, 0].sum() + c[:, p, 0].sum()), wins=w, losses=lo, draws=d, unfinished=u, score=s,
                             score_stderr=se))
    tot = c.sum(axis=(0, 1))
    s1, s1_se = _score(int(tot[1]), int(tot[3]), int(tot[1] + tot[2] + tot[3]))
    r, r_se = ratings(c)
    return dict(games=int(tot[0]), unfinished=int(tot[4]), policies=policies, pairs=out_pairs, score=score, score_stderr=score_se,
                by_seat=by_seat, seat1_score=s1, seat1_score_stderr=s1_se, ratings=r, rating_stderr=r_se)


def load_saved_actors(save_location: str = "training_models", actor_dir_name: str = "actor") -> list:
    """[(name, six get_weights() arrays)] of every actor a SkillshotLearner saved under save_location/actor_dir_name
    (``<start>_<end>_model.npz``), sorted by end epoch as load_actor_critic_models sorts them.  ``League([a for _, a in
    load_saved_actors(dir)], ...)`` rates every checkpoint of a run."""
    d = os.path.join(save_location, actor_dir_name)
    files = sorted((os.path.basename(f) for f in glob.glob(os.path.join(d, "*_model.npz"))), key=lambda x: int(x.split("_")[1]))
    out = []
    for f in files:
        with np.load(os.path.join(d, f)) as z:
            out.append((f[:-len("_model.npz")], [z[k] for k in z.files]))
    return out


class League:
    """``games_per_pair`` games of every scheduled pair of ``actors`` (2 .. 64 of them) on one GPU, one game per env.

    actors: flat vectors or the six get_weights() arrays each (see match.actor_vector; frames 1..20 inferred).  pairs:
    unordered pairs (i, j), i != j, each at most once, that connect all policies (default: the round robin).
    games_per_pair: even, >= 2; half of a pair's games seat i first, half j.  The vectors are COPIED at construction.
    precision "bf16": the tensor-core forwards; "f32": the exact float32 kernels.  speeds: None or the four per-env arrays
    of SkillshotEnvs.set_speeds (one entry per env, envs pair-major).
    """

    def __init__(self, actors, games_per_pair: int, pairs=None, device="cuda", precision: str = "bf16", tick_limit: int = 2000,
                 random_positions: bool = True, seed: int = 0, speeds=None, ticks_per_call: int = 64):
        if precision not in ("f32", "bf16"):
            raise ValueError("precision must be 'f32' (exact path) or 'bf16' (tensor cores)")
        vecs = [actor_vector(a) for a in actors]
        P = len(vecs)
        if not 2 <= P <= _lib.LEAGUE_MAX_POLICIES:
            raise ValueError("a league has 2..%d policies, got %d" % (_lib.LEAGUE_MAX_POLICIES, P))
        g = int(games_per_pair)
        if g < 2 or g % 2:
            raise ValueError("games_per_pair must be even and >= 2")
        if int(tick_limit) <= 0 or int(ticks_per_call) <= 0:
            raise ValueError("tick_limit and ticks_per_call must be positive")
        pairs = round_robin(P) if pairs is None else [(int(i), int(j)) for i, j in pairs]
        seen = set()
        for i, j in pairs:
            if not (0 <= i < P and 0 <= j < P) or i == j:
                raise ValueError("pair (%d, %d) is not two distinct policies of 0..%d" % (i, j, P - 1))
            if (min(i, j), max(i, j)) in seen:
                raise ValueError("pair (%d, %d) is scheduled twice" % (i, j))
            seen.add((min(i, j), max(i, j)))
        if not pairs or _components(P, pairs) != 1:
            raise ValueError("the schedule must connect all %d policies" % P)
        self.n_policies, self.pairs, self.games_per_pair = P, pairs, g
        self.frames = [f for _, f in vecs]
        self.precision, self.tick_limit, self.ticks_per_call = precision, int(tick_limit), int(ticks_per_call)
        n = self.n_envs = len(pairs) * g
        self.envs = SkillshotEnvs(n, device=device, random_positions=random_positions, seed=seed, reward_mode="none",
                                  tick_limit=self.tick_limit, auto_reset=False)
        self.device = dev = self.envs.device
        if speeds is not None:
            self.envs.set_speeds(*speeds)

        # seat tables on the host: policy of each seat, pair-major
        pol = np.empty((n, 2), np.int64)
        for k, (i, j) in enumerate(pairs):
            pol[k * g:k * g + g // 2] = (i, j)
            pol[k * g + g // 2:(k + 1) * g] = (j, i)
        # segment order: the 1-frame policies first (one forward launch), then the others, each in index order
        self.order = [p for p in range(P) if self.frames[p] == 1] + [p for p in range(P) if self.frames[p] > 1]
        seg_start = np.zeros(P + 1, np.int64)
        rows = np.empty((n, 2), np.int64)
        for s, p in enumerate(self.order):
            plays = (pol == p)                                   # [n][2]: at most one seat per env
            envs_p = np.nonzero(plays.any(1))[0]
            seg_start[s + 1] = seg_start[s] + envs_p.size
            seat = plays[envs_p, 1].astype(np.int64)
            rows[envs_p, seat] = seg_start[s] + np.arange(envs_p.size)
        assert seg_start[-1] == 2 * n and np.array_equal(np.sort(rows.ravel()), np.arange(2 * n))
        self.seg_start = seg_start
        self.seat_policy_host, self.seat_rows_host = pol.astype(np.uint8), rows.astype(np.int32)
        self.seat_rows = torch.from_numpy(self.seat_rows_host).to(dev)
        self.seat_policy = torch.from_numpy(self.seat_policy_host).to(dev)

        # parameter vectors in segment order, each 16-byte aligned
        self.param_stride = (max(v.size for v, _ in vecs) + 3) // 4 * 4
        flat = np.zeros(P * self.param_stride, np.float32)
        for s, p in enumerate(self.order):
            flat[s * self.param_stride:s * self.param_stride + vecs[p][0].size] = vecs[p][0]
        self.params = torch.from_numpy(flat).to(dev)

        obs = self.envs.observe()                                # [n][2][12]
        self.obs = torch.empty((2 * n, 12), dtype=torch.float32, device=dev)
        rr = self.seat_rows.long()
        self.obs[rr[:, 0]] = obs[:, 0]
        self.obs[rr[:, 1]] = obs[:, 1]
        self.act = torch.zeros((2 * n, 2), dtype=torch.float32, device=dev)
        tc = precision == "bf16"
        self.stacks = []
        for s, p in enumerate(self.order):
            f, m = self.frames[p], int(seg_start[s + 1] - seg_start[s])
            if f == 1:
                self.stacks.append(None)
                continue
            st = (torch.zeros(int(lib.ss_obs_stack_tc_bytes(m, f)), dtype=torch.uint8, device=dev) if tc
                  else torch.zeros((m, f, 12), dtype=torch.float32, device=dev))
            # the first observation fills every slot (FrameStackActor.push)
            ones = torch.ones(m, dtype=torch.uint8, device=dev)
            push = lib.ss_obs_stack_push_tc if tc else lib.ss_obs_stack_push
            with torch.cuda.device(dev):
                check(push(st.data_ptr(), m, f, 0, self.obs[int(seg_start[s]):].data_ptr(), ones.data_ptr(), 1, _stream(dev)),
                      "ss_obs_stack_push")
            self.stacks.append(st)
        self.head = 0
        self.ticks = 0
        a = self._args = _lib.LeagueArgs()
        self._seg = (ctypes.c_int64 * (P + 1))(*[int(v) for v in seg_start])
        self._frames = (ctypes.c_int * P)(*[self.frames[p] for p in self.order])
        self._stacks = (ctypes.c_void_p * P)(*[None if st is None else st.data_ptr() for st in self.stacks])
        a.state, a.n_envs, a.tick_limit = self.envs.state.data_ptr(), n, self.tick_limit
        a.speeds = None if self.envs.speeds is None else self.envs.speeds.data_ptr()
        a.status = self.envs.status.data_ptr()
        a.seat_rows, a.obs, a.act = self.seat_rows.data_ptr(), self.obs.data_ptr(), self.act.data_ptr()
        a.params, a.param_stride, a.n_policies = self.params.data_ptr(), self.param_stride, P
        a.seg_start = ctypes.cast(self._seg, ctypes.POINTER(ctypes.c_int64))
        a.frames = ctypes.cast(self._frames, ctypes.POINTER(ctypes.c_int))
        a.stacks = ctypes.cast(self._stacks, ctypes.POINTER(ctypes.c_void_p))
        a.tensor_cores = 1 if tc else 0
        ws = int(lib.ss_league_workspace_bytes(a))
        if ws < 0:
            raise ValueError("ss_league_workspace_bytes rejected the league's segments")
        self.workspace = torch.empty(max(ws, 16), dtype=torch.uint8, device=dev)
        a.workspace, a.workspace_bytes = self.workspace.data_ptr(), self.workspace.numel()
        self._counters = torch.zeros(P * P * 8, dtype=torch.int64, device=dev)
        self._host = torch.zeros(P * P * 8, dtype=torch.int64, pin_memory=True)

    def advance(self, n_ticks: int):
        """Enqueue n_ticks more league ticks (one ss_league_play call); reads nothing back."""
        self._args.head, self._args.n_ticks = self.head, int(n_ticks)
        with torch.cuda.device(self.device):
            check(lib.ss_league_play(self._args, _stream(self.device)), "ss_league_play")
        self.head += int(n_ticks)
        self.ticks += int(n_ticks)

    def counters(self) -> np.ndarray:
        """int64 [P][P][8] outcome counters of the games as they stand (ss_league_summary): cell (i, j) = the games with
        policy i in seat 1 and j in seat 2 {games, seat-1 wins, seat-2 wins, draws, unfinished, ticks of decided games}."""
        P = self.n_policies
        with torch.cuda.device(self.device):
            check(lib.ss_league_summary(self.envs.state.data_ptr(), self.n_envs, self.seat_policy.data_ptr(), P, self.tick_limit,
                                        self._counters.data_ptr(), _stream(self.device)), "ss_league_summary")
        self._host.copy_(self._counters)          # (synchronous: the host reads it next)
        return self._host.numpy().reshape(P, P, 8).copy()

    def play(self) -> dict:
        """Play until no game is unfinished, or tick_limit ticks, in calls of ticks_per_call ticks, and return:
        games, unfinished; policies[p] {games, wins, losses, draws, unfinished, score, score_stderr}; pairs [{pair, games,
        i_wins, j_wins, draws, unfinished, score (i's), score_stderr}]; score / score_stderr [P][P] (row i's score against
        column j, NaN where not scheduled); by_seat {(i, j): counts with i in seat 1}; seat1_score / seat1_score_stderr
        (the player-1 seat's pooled score: the seats are not symmetric); ratings / rating_stderr (see ratings())."""
        c = self.counters()
        while self.ticks < self.tick_limit and int(c[:, :, 4].sum()) > 0:
            self.advance(min(self.ticks_per_call, self.tick_limit - self.ticks))
            c = self.counters()
        self.envs.check_status()
        return summarize(c, self.pairs)
