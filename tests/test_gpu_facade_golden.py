"""The reference's per-tick caller sequence on the single-game facade, against the reference's own recorded answers.

SkillshotLearner.do_actions for both players, SkillshotGame.game_tick, get_state, prepare_states and
calculate_rewards_looking / _simple (SkillshotLearner.py:206-213, 304-315, 512-603), called through this package's
SkillshotLearner on skillshot_learning_b200.SkillshotGame views of device envs, tick by tick, for episodes of
tests/golden (recorded from the unmodified reference by oracle/gen_golden.py): every mutable field equal after every
tick, get_state features and prepare_states rows to 1e-12, rewards to 1e-12.  Unlike test_gpu_reference_callers this
needs no copy of the reference at run time."""
import contextlib
import io

import numpy as np
import pytest

from oracle import ref_harness
from tests import parity
from tests.helpers import load_golden

pytestmark = pytest.mark.gpu

EPISODES = 8          # per golden file: every call below is one launch plus a read-back


def _learner(game):
    from skillshot_learning_b200.learner import SkillshotLearner
    skl = object.__new__(SkillshotLearner)          # the caller surface only, no networks
    skl.game_environment = game
    skl.player_ids = (1, 2)
    skl.max_dist_normaliser = (2 * (250 ** 2)) ** 0.5
    return skl


def _want_state(g, i, t):
    return dict(px=[int(v) for v in g["px"][i, t]], py=[int(v) for v in g["py"][i, t]],
                prot=[float(v) for v in g["prot"][i, t]],
                qx=[int(v) for v in g["qx"][i, t]], qy=[int(v) for v in g["qy"][i, t]],
                qrot=[float(v) for v in g["qrot"][i, t]],
                cd=[int(v) for v in g["cd"][i, t]], age=[int(v) for v in g["age"][i, t]],
                valid=[int(v) for v in g["valid"][i, t]],
                ticks=int(g["ticks"][i, t]), live=int(g["live"][i, t]), winner=int(g["winner"][i, t]))


@pytest.mark.parametrize("name", ["kat", "lockstep_fixed", "lockstep_random", "close_hits"])
def test_caller_sequence_on_the_facade_matches_the_recorded_reference(name):
    from skillshot_learning_b200.game import SkillshotEnvs
    g = load_golden(name)
    envs = parity.start_from_golden(lambda n, **kw: SkillshotEnvs(n, device="cuda:0", **kw), g, reward_mode="none")
    n, T = g["actions"].shape[:2]
    episodes = range(min(n, EPISODES))
    terminals = 0
    for i in episodes:
        game = envs.game(i)
        skl = _learner(game)
        assert ref_harness.read_state(game) == _want_state(g, i, 0), (name, i)
        states = []
        with contextlib.redirect_stdout(io.StringIO()):
            for t in range(T):
                for pid in (1, 2):
                    skl.do_actions(pid, (float(g["actions"][i, t, pid - 1, 0]), float(g["actions"][i, t, pid - 1, 1])))
                game.game_tick()
                msg = f"{name} episode {i} t={t + 1}"
                assert ref_harness.read_state(game) == _want_state(g, i, t + 1), msg    # floats compared with ==
                sd = game.get_state()
                assert (sd["game_live"], sd["ticks"], sd["game_winner"]) == (
                    bool(g["live"][i, t + 1]), int(g["ticks"][i, t + 1]), int(g["winner"][i, t + 1])), msg
                feat = ref_harness.features_of(sd)[None]
                want = g["feat"][i, t + 1][None]
                st = {k: g[k][i:i + 1, t + 1] for k in ("qx", "qy", "px", "py", "valid", "qrot")}
                amb = parity.ambiguous_future_collision(st, want[..., 8], count=False)
                feat[..., 17] = np.where(amb, want[..., 17], feat[..., 17])
                parity.assert_features_close(feat, want, msg)
                states.append((sd, amb[0]))
        for pid in (1, 2):
            rows = np.array(skl.prepare_states([s for s, _ in states], pid), dtype=np.float64)
            want = g["obs"][i, 1:, pid - 1]
            amb = np.array([a[pid - 1] for _, a in states])
            rows[amb, 11] = want[amb, 11]
            np.testing.assert_array_equal(rows[:, 11], want[:, 11], err_msg=f"{name} {i} future-collision flag")
            np.testing.assert_allclose(rows, want, rtol=1e-12, atol=1e-12, err_msg=f"{name} {i} prepare_states")
        for fn, key in (("calculate_rewards_looking", "rew_looking"), ("calculate_rewards_simple", "rew_simple")):
            got = np.array([[r[1], r[2]] for r in getattr(skl, fn)([s for s, _ in states])], dtype=np.float64)
            np.testing.assert_allclose(got, g[key][i, 1:], rtol=1e-12, atol=1e-9, err_msg=f"{name} {i} {fn}")
        terminals += int(g["live"][i, -1] == 0)
    if name in ("kat", "close_hits"):
        assert terminals > 0          # games that end in a hit are among those replayed
