"""B200-native Skillshot hot path: batched SkillshotGame tick, rollout and DDPG
update as hand-written sm_100a kernels behind a C ABI (include/skillshot_b200.h).
Importing the package loads the CUDA library and fails if it has not been built."""
from . import _lib  # noqa: F401  (raises ImportError when libskillshot_b200.so is missing)
from .game import Player, Projectile, SkillshotEnvs, SkillshotGame, render_board  # noqa: F401

from .learner import ActorCritic, FrameStackActor, ReplayRing, SelfPlayTrainer, SkillshotLearner  # noqa: F401
from .match import Match  # noqa: F401
from .league import League, gauntlet, load_saved_actors, ratings, round_robin  # noqa: F401

__all__ = ["SkillshotEnvs", "SkillshotGame", "Player", "Projectile", "render_board",
           "ActorCritic", "FrameStackActor", "ReplayRing", "SelfPlayTrainer", "SkillshotLearner", "Match",
           "League", "round_robin", "gauntlet", "ratings", "load_saved_actors"]
