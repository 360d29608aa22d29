"""Head-to-head matches between two actors on one GPU (ss_match_play, include/skillshot_b200.h).

The self-play statistics (SelfPlayTrainer.progress) count how games of ONE policy against itself end; they measure the
game's seat asymmetry and episode lengths, not playing strength.  A :class:`Match` plays policy A against policy B:

* every env plays exactly one game from tick 0 (no auto-reset), to a hit or to ``tick_limit`` ticks, so no outcome is
  sampled by its length;
* both policies play both seats -- check_collision tests player 1 first and a double hit records id 1, so the seats are
  not symmetric -- and the result is also reported per seat;
* ``winner_id`` is the id of the player that was HIT (SkillshotGame.py:77): an A win is a game in which B was hit.

The policies act deterministically (no parameter or action noise); the variety comes from the Philox start positions.
"""
from __future__ import annotations

import math
from typing import Optional

import numpy as np
import torch

from . import _lib
from ._lib import lib, check
from .game import SkillshotEnvs

def _actor_params(n: int) -> int:
    return int(lib.ss_actor_frames_params(n))


def actor_vector(actor):
    """(flat float32 numpy vector, frames) of an actor given as a flat vector of ss_actor_frames_params(F) values or as
    the six Keras get_weights() arrays [W1 (12 F, 256), b1, W2, b2, W3, b3] (what save_actor_critic_models writes).
    F is inferred from the length, or from W1's rows / 12; anything else raises ValueError."""
    if isinstance(actor, (list, tuple)):
        if len(actor) != 6:
            raise ValueError("an actor given as arrays must be the six get_weights() arrays, got %d" % len(actor))
        arrs = [a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a) for a in actor]
        rows = arrs[0].shape[0] if arrs[0].ndim == 2 else -1
        frames = rows // 12 if rows > 0 and rows % 12 == 0 else 0
        if not 1 <= frames <= _lib.MAX_FRAMES:
            raise ValueError("W1 must have 12 * frames rows (frames 1..20), got shape %s" % (arrs[0].shape,))
        want = [(12 * frames, 256), (256,), (256, 128), (128,), (128, 2), (2,)]
        for a, sh in zip(arrs, want):
            if tuple(a.shape) != sh:
                raise ValueError("actor array of shape %s where %s was expected" % (tuple(a.shape), sh))
        return np.concatenate([a.reshape(-1) for a in arrs]).astype(np.float32), frames
    flat = actor.detach().cpu().numpy() if torch.is_tensor(actor) else np.asarray(actor)
    if flat.ndim != 1:
        raise ValueError("an actor vector must be one-dimensional, got shape %s" % (flat.shape,))
    for frames in range(1, _lib.MAX_FRAMES + 1):
        if flat.size == _actor_params(frames):
            return flat.astype(np.float32), frames
    raise ValueError("%d values is no actor's parameter count (ss_actor_frames_params(1..20))" % flat.size)


def _block(c) -> dict:
    games, a_wins, b_wins, draws, unfinished, ticks = (int(v) for v in c[:6])
    decided = a_wins + b_wins
    return dict(games=games, a_wins=a_wins, b_wins=b_wins, draws=draws, unfinished=unfinished,
                score=(a_wins + draws / 2) / games if games else float("nan"),
                mean_ticks_decided=ticks / decided if decided else float("nan"))


def summarize(counters) -> dict:
    """The result dict of Match.play from the uint64 [2][8] counters of ss_match_summary (block 0: A is player 1).
    score = (a_wins + draws / 2) / games; score_stderr = the standard error of the mean of the per-game scores (1 for an A
    win, 1/2 for a draw, 0 otherwise), with the sample variance."""
    c = np.asarray(counters, dtype=np.int64).reshape(2, 8)
    out = _block(c[0] + c[1])
    g, mean = out["games"], out["score"]
    if g > 1:
        # per-game scores s in {1, 1/2, 0}: sum s^2 = a_wins + draws / 4
        var = ((out["a_wins"] + out["draws"] / 4) - g * mean * mean) / (g - 1)
        out["score_stderr"] = math.sqrt(max(var, 0.0) / g)
    else:
        out["score_stderr"] = float("nan")
    out["by_seat"] = {"a_player1": _block(c[0]), "a_player2": _block(c[1])}
    return out


def _stream(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


class Match:
    """``n_games`` games of actor A against actor B on one GPU, one game per env, Philox random (or fixed) starts.

    In env j < split A is player 1 and B player 2, in env j >= split the other way round (split defaults to n_games // 2).
    Both parameter vectors are COPIED at construction: training that continues afterwards does not change the match.
    precision "bf16": the tensor-core forwards; "f32": the exact float32 kernels.  speeds: None or the four per-env arrays
    of SkillshotEnvs.set_speeds.
    """

    def __init__(self, actor_a, actor_b, n_games: int, device="cuda", precision: str = "bf16", tick_limit: int = 2000,
                 random_positions: bool = True, seed: int = 0, split: Optional[int] = None, speeds=None,
                 ticks_per_call: int = 64):
        if precision not in ("f32", "bf16"):
            raise ValueError("precision must be 'f32' (exact path) or 'bf16' (tensor cores)")
        n = int(n_games)
        if n <= 0 or int(tick_limit) <= 0 or int(ticks_per_call) <= 0:
            raise ValueError("n_games, tick_limit and ticks_per_call must be positive")
        split = n // 2 if split is None else int(split)
        if not 0 <= split <= n:
            raise ValueError("split must lie in 0..n_games")
        va, fa = actor_vector(actor_a)
        vb, fb = actor_vector(actor_b)
        self.n_games, self.split, self.tick_limit = n, split, int(tick_limit)
        self.frames_a, self.frames_b, self.precision = fa, fb, precision
        self.ticks_per_call = int(ticks_per_call)
        self.envs = SkillshotEnvs(n, device=device, random_positions=random_positions, seed=seed, reward_mode="none",
                                  tick_limit=self.tick_limit, auto_reset=False)
        self.device = dev = self.envs.device
        if speeds is not None:
            self.envs.set_speeds(*speeds)
        # [A | B], each vector 16-byte aligned
        self.param_stride = (max(va.size, vb.size) + 3) // 4 * 4
        self.params = torch.zeros(2 * self.param_stride, dtype=torch.float32, device=dev)
        self.params[:va.size].copy_(torch.from_numpy(va))
        self.params[self.param_stride:self.param_stride + vb.size].copy_(torch.from_numpy(vb))
        # policy-major observations [2][n][12]: half 0 is A's (player 1's in env j < split), half 1 is B's
        obs = self.envs.observe()
        seat_a = torch.arange(n, device=dev) >= split                     # A's seat index (0 = player 1)
        ar = torch.arange(n, device=dev)
        self.obs = torch.stack([obs[ar, seat_a.long()], obs[ar, (~seat_a).long()]]).contiguous()
        self.act = torch.zeros((2, n, 2), dtype=torch.float32, device=dev)
        tc = precision == "bf16"
        self.stacks = []
        for p, f in enumerate((fa, fb)):
            if f == 1:
                self.stacks.append(None)
                continue
            st = (torch.zeros(int(lib.ss_obs_stack_tc_bytes(n, f)), dtype=torch.uint8, device=dev) if tc
                  else torch.zeros((n, f, 12), dtype=torch.float32, device=dev))
            # the first observation fills every slot (FrameStackActor.push)
            ones = torch.ones(n, dtype=torch.uint8, device=dev)
            push = lib.ss_obs_stack_push_tc if tc else lib.ss_obs_stack_push
            with torch.cuda.device(dev):
                check(push(st.data_ptr(), n, f, 0, self.obs[p].data_ptr(), ones.data_ptr(), 1, _stream(dev)), "ss_obs_stack_push")
            self.stacks.append(st)
        self.head = 0
        ws = int(lib.ss_match_workspace_bytes(n, fa, fb, 1 if tc else 0))
        self.workspace = torch.empty(max(ws, 16), dtype=torch.uint8, device=dev)
        self._counters = torch.zeros(_lib.MATCH_STATS, dtype=torch.int64, device=dev)
        self._host = torch.zeros(_lib.MATCH_STATS, dtype=torch.int64, pin_memory=True)
        self.ticks = 0
        a = self._args = _lib.MatchArgs()
        a.state, a.n_envs, a.split, a.tick_limit = self.envs.state.data_ptr(), n, split, self.tick_limit
        a.speeds = None if self.envs.speeds is None else self.envs.speeds.data_ptr()
        a.status = self.envs.status.data_ptr()
        a.obs, a.act, a.params, a.param_stride = self.obs.data_ptr(), self.act.data_ptr(), self.params.data_ptr(), self.param_stride
        a.frames_a, a.frames_b = fa, fb
        a.stack_a = None if self.stacks[0] is None else self.stacks[0].data_ptr()
        a.stack_b = None if self.stacks[1] is None else self.stacks[1].data_ptr()
        a.workspace, a.workspace_bytes, a.tensor_cores = self.workspace.data_ptr(), self.workspace.numel(), 1 if tc else 0

    def advance(self, n_ticks: int):
        """Enqueue n_ticks more match ticks (one ss_match_play call); reads nothing back."""
        self._args.head, self._args.n_ticks = self.head, int(n_ticks)
        with torch.cuda.device(self.device):
            check(lib.ss_match_play(self._args, _stream(self.device)), "ss_match_play")
        self.head += int(n_ticks)
        self.ticks += int(n_ticks)

    def counters(self) -> np.ndarray:
        """int64 [2][8] outcome counters of the games as they stand (ss_match_summary; 128 bytes read back)."""
        with torch.cuda.device(self.device):
            check(lib.ss_match_summary(self.envs.state.data_ptr(), self.n_games, self.split, self.tick_limit,
                                       self._counters.data_ptr(), _stream(self.device)), "ss_match_summary")
        self._host.copy_(self._counters)          # (synchronous: the host reads it next)
        return self._host.numpy().reshape(2, 8).copy()

    def play(self) -> dict:
        """Play until no game is unfinished, or tick_limit ticks, in calls of ticks_per_call ticks, and return the
        result: games, a_wins, b_wins, draws, unfinished, score, score_stderr, mean_ticks_decided and by_seat
        {"a_player1": ..., "a_player2": ...} (the same counts, score and mean length per seat)."""
        c = self.counters()
        while self.ticks < self.tick_limit and int(c[:, 4].sum()) > 0:
            self.advance(min(self.ticks_per_call, self.tick_limit - self.ticks))
            c = self.counters()
        self.envs.check_status()
        return summarize(c)
