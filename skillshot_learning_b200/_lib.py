"""ctypes binding of libskillshot_b200.so (the C ABI of include/skillshot_b200.h).

There is no CPU fallback: if the CUDA library is missing, importing this module
raises.  Build it with `python -m skillshot_learning_b200.build`.
"""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libskillshot_b200.so")

# constants of include/skillshot_b200.h
STATE_BYTES_PER_ENV = 64
NUM_FEATURES = 18
NUM_OBS = 12
EXPORT_INTS = 17
REWARD_NONE, REWARD_LOOKING, REWARD_TERMINAL, REWARD_SIMPLE = 0, 1, 2, 3
RESET_FIXED, RESET_RANDOM, RESET_GIVEN = 0, 1, 2
STEP_OBS_EVERY_TICK = 1
STEP_EPISODE_STATS = 2
EPISODE_STATS = 72
STATUS_NAN = 1
STATUS_PEER_TIMEOUT = 2
STATUS_ROLLOUT_TIMEOUT = 4
(OP_MOVE_DIRECTION_FLOAT, OP_MOVE_LOOK_FLOAT, OP_SHOOT, OP_MOVE_FORWARDS, OP_MOVE_BACKWARDS,
 OP_LOOK_LEFT, OP_LOOK_RIGHT, OP_GAME_TICK) = range(8)

_vp, _i64, _i32, _u64, _f64 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_uint64, ctypes.c_double
_f32 = ctypes.c_float

# learner constants of include/skillshot_b200.h
DIM_STATE, DIM_ACTION, HIDDEN1, HIDDEN2 = 12, 2, 256, 128
ACTOR_PARAMS, CRITIC_PARAMS = 36482, 36609
PEER_MAX_WORLD, PEER_HANDLE_BYTES = 8, 64

_u32 = ctypes.c_uint32


PAIR_MAIL_EMPTY = 0x7fc0dead      # SS_PAIR_MAIL_EMPTY
MATCH_STATS = 16                  # SS_MATCH_STATS: uint64 [2][8] of ss_match_summary
MAX_FRAMES = 20                   # SS_MAX_FRAMES
LEAGUE_MAX_POLICIES = 64          # SS_LEAGUE_MAX_POLICIES
STATUS_SEAT_RANGE = 8             # SS_STATUS_SEAT_RANGE
POOL_STATS = 8                    # uint64 counters per opponent of ss_env_step_pool / ss_pool_rollout
TAG_TARGET_NOISE = 5              # SS_TAG_TARGET_NOISE: Philox tag of the TD3 target policy smoothing


def td3_tc_workspace_bytes(n: int) -> int:
    """SS_TD3_TC_WORKSPACE_BYTES(n): the workspace of ss_td3_targets_tc with two critics."""
    return (n * 8 + 15) // 16 * 16 + 2 * ((n * 4 + 15) // 16 * 16)


class DdpgUpdateArgs(ctypes.Structure):
    """struct ss_ddpg_update_args of include/skillshot_b200.h (same field order)."""
    _fields_ = ([(k, _vp) for k in ("ring_obs", "ring_act", "ring_reward", "ring_next_obs", "ring_done")] +
                [("capacity", _i64), ("size", _i64), ("replay_seed", _u64), ("replay_counter", _u64), ("batch", _i64)] +
                [(k, _vp) for k in ("obs", "act", "reward", "next_obs", "done", "indices", "y", "actor", "critic",
                                    "target_actor", "target_critic", "m_actor", "v_actor", "m_critic", "v_critic",
                                    "grad_actor", "grad_critic", "stats")] +
                [(k, _f32) for k in ("gamma", "tau", "lr_actor", "lr_critic", "beta1", "beta2", "eps", "dropout_rate")] +
                [("seed", _u64), ("counter", _u64), ("step_critic", _i64), ("step_actor", _i64), ("n_global", _i64),
                 ("row_offset", _i64), ("workspace", _vp), ("workspace_bytes", _i64), ("tensor_cores", _i32),
                 ("world", _i32), ("rank", _i32), ("peer_bases", _vp), ("peer_capacity", _i64), ("epoch", _u32),
                 ("done_counter", _vp), ("status", _vp), ("pair_mail", _vp), ("sample_early", _i32)])


class MatchArgs(ctypes.Structure):
    """struct ss_match_args of include/skillshot_b200.h (same field order)."""
    _fields_ = [("state", _vp), ("n_envs", _i64), ("split", _i64), ("tick_limit", _i64), ("speeds", _vp), ("status", _vp),
                ("obs", _vp), ("act", _vp), ("params", _vp), ("param_stride", _i64), ("frames_a", _i32), ("frames_b", _i32),
                ("stack_a", _vp), ("stack_b", _vp), ("head", _i64), ("workspace", _vp), ("workspace_bytes", _i64),
                ("tensor_cores", _i32), ("n_ticks", _i32)]


class LeagueArgs(ctypes.Structure):
    """struct ss_league_args of include/skillshot_b200.h (same field order)."""
    _fields_ = [("state", _vp), ("n_envs", _i64), ("tick_limit", _i64), ("speeds", _vp), ("status", _vp), ("seat_rows", _vp),
                ("obs", _vp), ("act", _vp), ("params", _vp), ("param_stride", _i64), ("n_policies", _i32),
                ("seg_start", ctypes.POINTER(_i64)), ("frames", ctypes.POINTER(_i32)), ("stacks", ctypes.POINTER(_vp)),
                ("head", _i64), ("workspace", _vp), ("workspace_bytes", _i64), ("tensor_cores", _i32), ("n_ticks", _i32)]


class PoolRolloutArgs(ctypes.Structure):
    """struct ss_pool_rollout_args of include/skillshot_b200.h (same field order)."""
    _fields_ = ([("state", _vp), ("n_envs", _i64), ("pool_envs", _i64), ("n_opponents", _i32), ("params", _vp), ("opp_params", _vp),
                 ("opp_param_stride", _i64)] +
                [(k, _vp) for k in ("obs", "act", "reward", "opp_obs", "opp_act", "done", "winner", "ring_obs", "ring_act",
                                    "ring_reward", "ring_next_obs", "ring_done")] +
                [("capacity", _i64), ("write_pos", _i64), ("n_ticks", _i32), ("param_noise_sd", _f32), ("noise_group", _i64),
                 ("action_noise_sd", _f32), ("tensor_cores", _i32), ("reward_mode", _i32), ("tick_limit", _i64),
                 ("reset_mode", _i32), ("env_seed", _u64), ("env_counter", _u64), ("noise_seed", _u64), ("noise_counter", _u64),
                 ("speeds", _vp), ("status", _vp), ("step_flags", _i32), ("pool_stats", _vp)])


class PoolRolloutFramesArgs(ctypes.Structure):
    """struct ss_pool_rollout_frames_args of include/skillshot_b200.h (same field order): ss_pool_rollout_args' fields, then
    the histories."""
    _fields_ = PoolRolloutArgs._fields_ + [
        ("frames", _i32), ("stack_tc", _vp), ("stack32", _vp), ("rows", _vp), ("head", _i64),
        ("opp_frames", ctypes.POINTER(_i32)), ("opp_stacks", ctypes.POINTER(_vp)), ("workspace", _vp), ("workspace_bytes", _i64),
        ("opp_envs", ctypes.POINTER(_i64))]


# name -> (restype, argtypes); every symbol the header declares
SIGNATURES = {
    "ss_version": (_i32, []),
    "ss_state_bytes": (_i64, [_i64]),
    "ss_env_reset": (_i32, [_vp, _i64, _vp, _i32, _vp, _u64, _u64, _vp]),
    "ss_env_step": (_i32, [_vp, _i64, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i64, _i32, _i32, _u64, _u64,
                            _vp, _vp, _i32, _vp]),
    "ss_env_step_ring": (_i32, [_vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i64, _i32, _i32, _u64, _u64,
                                 _vp, _vp, _i32, _vp]),
    "ss_env_step_packed": (_i32, [_vp, _i64, _vp, _vp, _i32, _i64, _i32, _i32, _u64, _u64, _vp, _vp]),
    "ss_env_features": (_i32, [_vp, _i64, _vp, _vp, _vp, _vp, _vp]),
    "ss_env_export": (_i32, [_vp, _i64, _i64, _i64, _vp, _vp, _vp]),
    "ss_env_import": (_i32, [_vp, _i64, _i64, _i64, _vp, _vp, _vp]),
    "ss_env_apply": (_i32, [_vp, _i64, _i64, _i32, _i32, _f64, _vp, _vp, _vp]),
    "ss_learner_workspace_bytes": (_i64, []),
    "ss_actor_forward": (_i32, [_vp, _vp, _vp, _i64, _f32, _i64, _f32, _u64, _u64, _vp]),
    "ss_actor_forward_tc": (_i32, [_vp, _vp, _vp, _i64, _f32, _i64, _f32, _u64, _u64, _vp]),
    "ss_actor_forward_step_tc": (_i32, [_vp, _vp, _vp, _i64, _f32, _i64, _f32, _u64, _u64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32,
                                         _i64, _i32, _u64, _u64, _vp, _i32, _vp]),
    "ss_critic_forward_tc": (_i32, [_vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _f32, _vp, _vp]),
    "ss_critic_grad_tc": (_i32, [_vp, _vp, _vp, _vp, _vp, _f32, _u64, _u64, _i64, _i64, _i64, _vp, _vp, _vp, _i64, _vp]),
    "ss_actor_grad_tc": (_i32, [_vp, _vp, _vp, _i64, _vp, _vp, _vp, _i64, _vp]),
    "ss_actor_grad_tc_staged": (_i32, [_vp, _vp, _vp, _i64, _vp, _vp, _vp, _i64, _i32, _vp]),
    "ss_ddpg_targets_tc": (_i32, [_vp, _vp, _vp, _vp, _vp, _f32, _vp, _i64, _vp, _i64, _vp]),
    "ss_set_dependent_launch": (_i32, [_i32]),
    "ss_actor_critic_forward_tc": (_i32, [_vp, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _f32, _vp, _vp, _vp]),
    "ss_actor_grad_tc_paired": (_i32, [_vp, _vp, _vp, _i64, _vp, _vp, _vp, _i64, _i32, _vp, _vp]),
    "ss_ddpg_targets_tc_paired": (_i32, [_vp, _vp, _vp, _vp, _vp, _f32, _vp, _i64, _vp, _i64, _vp, _vp]),
    "ss_peer_bytes": (_i64, [_i32, _i64]),
    "ss_peer_alloc": (_i32, [_i32, _i64, _vp]),
    "ss_peer_free": (_i32, [_vp]),
    "ss_peer_export": (_i32, [_vp, _vp]),
    "ss_peer_import": (_i32, [_vp, _vp]),
    "ss_peer_close": (_i32, [_vp]),
    "ss_peer_reduce_push": (_i32, [_vp, _i32, _i32, _vp, _vp, _i32, _i32, _i64, ctypes.c_uint32, _vp, _vp]),
    "ss_peer_adam_tf": (_i32, [_vp, _i32, _i64, ctypes.c_uint32, _vp, _vp, _vp, _vp, _vp, _i64, _i64,
                                _f32, _f32, _f32, _f32, _f32, _f32, _vp, _vp]),
    "ss_peer_reduce_adam_tf": (_i32, [_vp, _i32, _i32, _vp, _vp, _i32, _i32, _i64, ctypes.c_uint32, _vp, _vp, _vp, _vp, _vp, _i64,
                                       _f32, _f32, _f32, _f32, _f32, _f32, _vp, _vp]),
    "ss_selfplay_rollout": (_i32, [_vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i32,
                                    _f32, _i64, _f32, _i32, _i32, _i64, _i32, _u64, _u64, _u64, _u64, _vp, _vp, _i32,
                                    _vp]),
    "ss_selfplay_rollout2": (_i32, [_vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i32,
                                     _f32, _i64, _f32, _i32, _i32, _i64, _i32, _u64, _u64, _u64, _u64, _vp, _vp, _i32,
                                     _vp, _vp, _vp]),
    "ss_actor_forward_tc_signal": (_i32, [_vp, _vp, _vp, _i64, _f32, _i64, _f32, _u64, _u64, _vp, _vp, _vp, _vp]),
    "ss_env_step_tiles": (_i32, [_vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i64, _i32, _u64, _u64, _vp, _i32, _vp,
                                  _i64, _i32, _vp]),
    "ss_actor_frames_params": (_i64, [_i32]),
    "ss_obs_stack_push": (_i32, [_vp, _i64, _i32, _i64, _vp, _vp, _i32, _vp]),
    "ss_param_noise_groups": (_i32, [_vp, _vp, _i64, _i64, _i64, _f32, _u64, _u64, _vp]),
    "ss_actor_forward_frames": (_i32, [_vp, _i64, _i64, _vp, _i32, _i64, _vp, _i64, _vp]),
    "ss_actor_frames_tc_workspace_bytes": (_i64, [_i64, _i64]),
    "ss_obs_stack_tc_bytes": (_i64, [_i64, _i32]),
    "ss_obs_stack_push_tc": (_i32, [_vp, _i64, _i32, _i64, _vp, _vp, _i32, _vp]),
    "ss_actor_forward_frames_tc": (_i32, [_vp, _i64, _i64, _vp, _i32, _i64, _vp, _i64, _vp, _i64, _vp]),
    "ss_critic_frames_params": (_i64, [_i32]),
    "ss_learner_frames_workspace_bytes": (_i64, [_i32]),
    "ss_obs_stack_ordered": (_i32, [_vp, _i64, _i32, _i64, _vp, _vp]),
    "ss_critic_forward_frames": (_i32, [_vp, _i32, _vp, _vp, _vp, _i64, _vp]),
    "ss_ddpg_targets_frames": (_i32, [_vp, _vp, _i32, _vp, _vp, _vp, _f32, _vp, _i64, _vp]),
    "ss_critic_grad_frames": (_i32, [_vp, _i32, _vp, _vp, _vp, _vp, _f32, _u64, _u64, _i64, _i64, _i64, _vp, _vp, _vp, _i64, _vp]),
    "ss_actor_grad_frames": (_i32, [_vp, _vp, _i32, _vp, _i64, _vp, _vp, _vp, _i64, _vp]),
    "ss_learner_frames_tc_workspace_bytes": (_i64, [_i32, _i64]),
    "ss_critic_forward_frames_tc": (_i32, [_vp, _i32, _vp, _vp, _vp, _vp, _i64, _vp, _i64, _vp]),
    "ss_ddpg_targets_frames_tc": (_i32, [_vp, _vp, _i32, _vp, _vp, _vp, _f32, _vp, _i64, _vp, _i64, _vp]),
    "ss_critic_grad_frames_tc": (_i32, [_vp, _i32, _vp, _vp, _vp, _vp, _f32, _u64, _u64, _i64, _i64, _i64, _vp, _vp, _vp, _i64,
                                         _vp]),
    "ss_actor_grad_frames_tc": (_i32, [_vp, _vp, _i32, _vp, _i64, _vp, _vp, _vp, _i64, _vp]),
    "ss_td3_targets_frames": (_i32, [_vp, _vp, _vp, _i32, _vp, _vp, _vp, _f32, _f32, _f32, _u64, _u64, _i64, _vp, _i64, _vp, _i64,
                                      _vp]),
    "ss_td3_targets_tc": (_i32, [_vp, _vp, _vp, _vp, _vp, _vp, _f32, _f32, _f32, _u64, _u64, _i64, _vp, _i64, _vp, _i64, _vp]),
    "ss_td3_targets_frames_tc": (_i32, [_vp, _vp, _vp, _i32, _vp, _vp, _vp, _f32, _f32, _f32, _u64, _u64, _i64, _vp, _i64, _vp,
                                         _i64, _vp]),
    "ss_replay_push_frames": (_i32, [_vp, _vp, _vp, _vp, _vp, _i64, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _i32, _i64, _vp]),
    "ss_replay_sample_frames": (_i32, [_vp, _vp, _vp, _vp, _vp, _i64, _i64, _i32, _vp, _u64, _u64, _i64,
                                        _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "ss_param_noise": (_i32, [_vp, _vp, _i64, _f32, _u64, _u64, _u64, _vp]),
    "ss_critic_forward": (_i32, [_vp, _vp, _vp, _vp, _i64, _vp]),
    "ss_ddpg_targets": (_i32, [_vp, _vp, _vp, _vp, _vp, _f32, _vp, _i64, _vp]),
    "ss_critic_grad": (_i32, [_vp, _vp, _vp, _vp, _vp, _f32, _u64, _u64, _i64, _i64, _i64, _vp, _vp, _vp, _i64, _vp]),
    "ss_actor_grad": (_i32, [_vp, _vp, _vp, _i64, _vp, _vp, _vp, _i64, _vp]),
    "ss_adam_tf": (_i32, [_vp, _vp, _vp, _vp, _vp, _i64, _i64, _f32, _f32, _f32, _f32, _f32, _f32, _vp]),
    "ss_reduce_adam_tf": (_i32, [_vp, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _f32, _f32, _f32, _f32, _f32, _f32, _vp]),
    "ss_replay_push": (_i32, [_vp, _vp, _vp, _vp, _vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _i32, _i64, _vp]),
    "ss_ddpg_update": (_i32, [ctypes.POINTER(DdpgUpdateArgs), _vp]),
    "ss_probe_rates": (_i32, [_vp, _vp, _vp]),
    "ss_env_step_match": (_i32, [_vp, _i64, _i64, _vp, _vp, _i64, _vp, _vp, _vp]),
    "ss_actor_forward_groups_tc": (_i32, [_vp, _i64, _i64, _vp, _vp, _i64, _vp]),
    "ss_match_summary": (_i32, [_vp, _i64, _i64, _i64, _vp, _vp]),
    "ss_match_workspace_bytes": (_i64, [_i64, _i32, _i32, _i32]),
    "ss_match_play": (_i32, [ctypes.POINTER(MatchArgs), _vp]),
    "ss_env_step_seated": (_i32, [_vp, _i64, _vp, _i64, _vp, _vp, _i64, _vp, _vp, _vp]),
    "ss_actor_forward_segments_tc": (_i32, [_vp, _i64, _vp, _i32, _vp, _vp, _vp]),
    "ss_league_summary": (_i32, [_vp, _i64, _vp, _i32, _i64, _vp, _vp]),
    "ss_league_workspace_bytes": (_i64, [ctypes.POINTER(LeagueArgs)]),
    "ss_league_play": (_i32, [ctypes.POINTER(LeagueArgs), _vp]),
    "ss_env_step_pool": (_i32, [_vp, _i64, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i64, _i32, _u64, _u64,
                                 _vp, _i32, _vp, _vp]),
    "ss_env_step_pool_blocks": (_i32, [_vp, _i64, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i64, _i32, _u64,
                                        _u64, _vp, _i32, _vp, ctypes.POINTER(_i64), _vp]),
    "ss_pool_restart": (_i32, [_vp, _i64, _i64, _i32, ctypes.POINTER(_i64), _i32, _u64, _u64, _vp, _vp, _vp, _vp]),
    "ss_pool_rollout": (_i32, [ctypes.POINTER(PoolRolloutArgs), _vp]),
    "ss_obs_stack_push_pool": (_i32, [_vp, _vp, _i64, _i64, _i32, _i64, _vp, _vp, _vp, _vp, _vp]),
    "ss_pool_rollout_frames_workspace_bytes": (_i64, [ctypes.POINTER(PoolRolloutFramesArgs)]),
    "ss_pool_rollout_frames": (_i32, [ctypes.POINTER(PoolRolloutFramesArgs), _vp]),
    "ss_env_step_pool_speeds": (_i32, [_vp, _i64, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i64, _i32, _u64,
                                        _u64, _vp, _i32, _vp, ctypes.POINTER(_i64), _vp, _vp]),
    "ss_pool_rollout_speeds": (_i32, [ctypes.POINTER(PoolRolloutFramesArgs), _vp]),
    "ss_replay_sample": (_i32, [_vp, _vp, _vp, _vp, _vp, _i64, _i64, _vp, _u64, _u64, _i64,
                                 _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
}


class SkillshotLibraryError(RuntimeError):
    pass


def _load() -> ctypes.CDLL:
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "skillshot_learning_b200: %s is missing -- build the CUDA library with "
            "`python -m skillshot_learning_b200.build` (there is no CPU fallback)" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the library is stale
        fn.restype, fn.argtypes = res, args
    return lib


lib = _load()


def check(rc: int, what: str) -> None:
    if rc != 0:
        raise SkillshotLibraryError("%s failed with code %d (%s)" % (
            what, rc, {-1: "invalid argument", -2: "CUDA error"}.get(rc, "unknown")))
