// ss_pool.cu -- ss_pool_rollout / ss_pool_rollout_frames / ss_pool_rollout_speeds: n training ticks of the self-play
// learner with part of its envs played against a pool of frozen opponents, from one host call (include/skillshot_b200.h,
// "training against a pool").
//
// A tick is the learner's forward over its L rows, the opponents' forwards over their M rows, ss_env_step_pool and, for
// the networks that read a history of frames, the push of the newest observations.  Every kernel is an existing entry
// point; this file checks the arguments before anything is enqueued and lays the learner's rows into the replay ring as
// ss_selfplay_rollout does.  ss_pool_rollout is the case where every network has one frame; ss_pool_rollout_speeds steps
// the envs with ss_env_step_pool_speeds and is otherwise the same launches.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/skillshot_b200.h"
#include "ss_launch.cuh"
#include "ss_pool_blocks.cuh"

namespace {

typedef ss_pool_rollout_frames_args Args;

int opp_frames(const Args &R, int k) { return R.opp_frames ? R.opp_frames[k] : 1; }

// the learner's noisy parameter vectors: one per noise group, 16-byte aligned (as FrameStackActor.forward lays them out)
bool learner_noisy(const Args &R) { return R.frames > 1 && R.param_noise_sd > 0.f; }
int64_t noisy_stride(const Args &R) { return (ss_actor_frames_params(R.frames) + 3) / 4 * 4; }
int64_t noise_groups(const Args &R, int64_t L) { return (L + R.noise_group - 1) / R.noise_group; }

// the block starts B_0 .. B_K of opponent k's pool envs (and so of its rows); false: an invalid layout or block table
// (a table also needs M < 2^31, the step's 32-bit table).  M = 0 takes no table.
bool block_starts(const Args &R, int64_t *start) {
    const int64_t M = R.pool_envs;
    if (M == 0) return !R.opp_envs;
    if (R.opp_envs && M > 0x7fffffff) return false;
    return sspool::block_starts(M, R.n_opponents, R.opp_envs, start);
}

// -1: the layout, frame counts or noise settings are invalid; else the workspace bytes: the learner's noisy vectors, then
// the frame-stacked tensor-core forward's layer-1 tiles for the largest of its calls (they run one after the other)
int64_t workspace_bytes(const Args &R) {
    const int64_t n = R.n_envs, M = R.pool_envs, K = R.n_opponents;
    if (n <= 0 || M < 0 || M > n || R.frames < 1 || R.frames > SS_MAX_FRAMES) return -1;
    int64_t start[SS_LEAGUE_MAX_POLICIES + 1];
    if (!block_starts(R, start)) return -1;
    if (R.param_noise_sd > 0.f && (R.noise_group <= 0 || (R.tensor_cores && R.noise_group % 128 != 0))) return -1;
    for (int k = 0; k < K && M > 0; ++k)
        if (opp_frames(R, k) < 1 || opp_frames(R, k) > SS_MAX_FRAMES) return -1;
    const int64_t L = 2 * (n - M) + M;
    int64_t noisy = 0, tiles = 0;
    if (learner_noisy(R)) {
        if (noise_groups(R, L) > 65535) return -1;            // ss_param_noise_groups' grid
        noisy = noise_groups(R, L) * noisy_stride(R) * 4;
    }
    if (!R.tensor_cores) return noisy;
    if (R.frames > 1) tiles = ss_actor_frames_tc_workspace_bytes(L, learner_noisy(R) ? R.noise_group : 0);
    for (int k = 0; k < K && M > 0; ++k) {
        if (opp_frames(R, k) == 1) continue;
        const int64_t b = ss_actor_frames_tc_workspace_bytes(start[k + 1] - start[k], 0);
        if (b > tiles) tiles = b;
    }
    return noisy + tiles;
}

// speeds: the env step is ss_env_step_pool_speeds (R.speeds required), else ss_env_step_pool(_blocks) (R.speeds NULL)
int rollout(const Args &R, bool speeds, void *stream) {
    const int64_t n = R.n_envs, M = R.pool_envs, K = R.n_opponents;
    if (!R.state || !R.params || !R.obs || !R.act || !R.reward || !R.done || !R.winner || n <= 0 || R.n_ticks <= 0)
        return SS_ERR_INVALID_ARG;
    if (M < 0 || M > n) return SS_ERR_INVALID_ARG;
    int64_t start[SS_LEAGUE_MAX_POLICIES + 1];
    if (!block_starts(R, start)) return SS_ERR_INVALID_ARG;
    if (R.frames < 1 || R.frames > SS_MAX_FRAMES || R.head < 0) return SS_ERR_INVALID_ARG;
    if (M > 0) {
        if (!R.opp_params || !R.opp_obs || !R.opp_act) return SS_ERR_INVALID_ARG;
        if ((R.opp_param_stride & 3) || R.opp_param_stride < 0) return SS_ERR_INVALID_ARG;
        for (int k = 0; k < K; ++k) {
            const int f = opp_frames(R, k);
            if (f < 1 || f > SS_MAX_FRAMES || (K > 1 && R.opp_param_stride < ss_actor_frames_params(f))) return SS_ERR_INVALID_ARG;
            if (f > 1 && (!R.opp_stacks || !R.opp_stacks[k] || ((uintptr_t)R.opp_stacks[k] & 15))) return SS_ERR_INVALID_ARG;
        }
    }
    if (speeds ? (!R.speeds || ((uintptr_t)R.speeds & 15)) : R.speeds != nullptr) return SS_ERR_INVALID_ARG;
    if (R.reward_mode != SS_REWARD_NONE && R.reward_mode != SS_REWARD_LOOKING && R.reward_mode != SS_REWARD_TERMINAL) return SS_ERR_INVALID_ARG;
    if (R.reset_mode != SS_RESET_FIXED && R.reset_mode != SS_RESET_RANDOM) return SS_ERR_INVALID_ARG;
    if (R.param_noise_sd < 0.f || R.action_noise_sd < 0.f) return SS_ERR_INVALID_ARG;
    if (R.param_noise_sd > 0.f && (R.noise_group <= 0 || (R.tensor_cores && R.noise_group % 128 != 0))) return SS_ERR_INVALID_ARG;
    if ((((uintptr_t)R.state | (uintptr_t)R.params | (uintptr_t)R.obs | (uintptr_t)R.opp_params | (uintptr_t)R.opp_obs |
          (uintptr_t)R.ring_obs | (uintptr_t)R.ring_next_obs) & 15) ||
        (((uintptr_t)R.act | (uintptr_t)R.opp_act | (uintptr_t)R.ring_act | (uintptr_t)R.pool_stats) & 7) ||
        (((uintptr_t)R.reward | (uintptr_t)R.ring_reward | (uintptr_t)R.status) & 3))
        return SS_ERR_INVALID_ARG;
    if (R.status && (R.step_flags & SS_STEP_EPISODE_STATS) && ((uintptr_t)R.status & 7)) return SS_ERR_INVALID_ARG;
    const int F = R.frames;
    if (F > 1) {
        // the frame-stacked forwards take no action noise
        if (!R.stack32 || !R.rows || (R.tensor_cores && !R.stack_tc) || R.action_noise_sd != 0.f) return SS_ERR_INVALID_ARG;
        if (((uintptr_t)R.stack32 | (uintptr_t)R.rows | (uintptr_t)R.stack_tc) & 15) return SS_ERR_INVALID_ARG;
    }
    const int64_t need = workspace_bytes(R);
    if (need < 0) return SS_ERR_INVALID_ARG;
    if (need > 0 && (!R.workspace || R.workspace_bytes < need || ((uintptr_t)R.workspace & 15))) return SS_ERR_INVALID_ARG;
    const int64_t S = n - M, L = 2 * S + M, w = 12 * (int64_t)F;
    const bool ring = R.ring_obs != nullptr;
    // the transitions are produced in place (see ss_selfplay_rollout: one segment of L rows per tick, and with a single
    // segment the second observation copy would overwrite the rows the actor has just read)
    if (ring && (!R.ring_act || !R.ring_reward || !R.ring_next_obs || !R.ring_done || R.capacity <= 0 || R.capacity % L != 0 ||
                 R.write_pos < 0 || R.write_pos >= R.capacity || R.write_pos % L != 0 || (R.capacity / L < 2 && R.n_ticks != 1)))
        return SS_ERR_INVALID_ARG;

    cudaStream_t st = (cudaStream_t)stream;
    const int64_t segs = ring ? R.capacity / L : 1;
    int64_t seg = ring ? R.write_pos / L : 0;
    if (ring && cudaMemcpyAsync(R.ring_obs + seg * L * w, F > 1 ? R.rows : R.obs, (size_t)(L * w * 4), cudaMemcpyDeviceToDevice, st) !=
                    cudaSuccess)
        return SS_ERR_CUDA;
    int64_t seg_rows[SS_LEAGUE_MAX_POLICIES];
    for (int k = 0; k < K && M > 0; ++k) seg_rows[k] = start[k + 1] - start[k];
    float *noisy = (float *)R.workspace;
    void *tiles = learner_noisy(R) ? (void *)(noisy + noise_groups(R, L) * noisy_stride(R)) : R.workspace;
    const int64_t tile_bytes = need - (learner_noisy(R) ? noise_groups(R, L) * noisy_stride(R) * 4 : 0);
    auto opp_prm = [&](int k) { return R.opp_params + k * R.opp_param_stride; };
    // The launches of a tick form the dependent-launch chain of ss_selfplay_rollout (ss_launch.cuh) where they take part in
    // it (the 1-frame forwards and the env step; the frame-stacked kernels are ordinary launches).  The 1-frame learner's
    // forward stages its parameters ahead of its wait from the second tick on (its predecessor, the env step or a history
    // push, does not write them); the opponents' segment forward always does (no predecessor writes the opponents' vectors).
    const int kOn = (R.tensor_cores && sslaunch::chain_enabled()) ? sslaunch::kPdlOn : sslaunch::kPdlOff;
    sslaunch::PdlScope scope(kOn);
    const int kEarly = kOn ? (sslaunch::kPdlOn | sslaunch::kPdlEarlyWeights) : kOn;
    for (int t = 0; t < R.n_ticks; ++t, seg = (seg + 1) % segs) {
        const int64_t head = R.head + t, nseg = (seg + 1) % segs;
        const bool last = t + 1 == R.n_ticks;
        float *o = ring ? R.ring_obs + seg * L * w : R.obs, *a = ring ? R.ring_act + seg * L * 2 : R.act;
        float *o_next = !ring ? R.obs : !last ? R.ring_obs + nseg * L * 12 : R.obs;
        sslaunch::pdl_mode() = t > 0 ? kEarly : kOn;
        const uint64_t nc = R.noise_counter + (uint64_t)t;
        int rc = SS_OK;
        if (F > 1) {
            const float *p = R.params;
            int64_t stride = 0;
            if (learner_noisy(R)) {
                rc = ss_param_noise_groups(R.params, noisy, ss_actor_frames_params(F), noise_groups(R, L), noisy_stride(R), R.param_noise_sd,
                                           R.noise_seed, nc, stream);
                if (rc != SS_OK) return rc;
                p = noisy;
                stride = noisy_stride(R);
            }
            rc = R.tensor_cores ? ss_actor_forward_frames_tc(p, stride, R.noise_group, R.stack_tc, F, head, a, L, tiles, tile_bytes, stream)
                                : ss_actor_forward_frames(p, stride, R.noise_group, R.stack32, F, head, a, L, stream);
        } else {
            rc = R.tensor_cores ? ss_actor_forward_tc(R.params, o, a, L, R.param_noise_sd, R.noise_group, R.action_noise_sd, R.noise_seed,
                                                      nc, stream)
                                : ss_actor_forward(R.params, o, a, L, R.param_noise_sd, R.noise_group, R.action_noise_sd, R.noise_seed,
                                                   nc, stream);
        }
        if (rc != SS_OK) return rc;
        sslaunch::pdl_mode() = kEarly;
        for (int k = 0; k < K && M > 0 && rc == SS_OK;) {
            const int64_t b = seg_rows[k];
            float *oo = R.opp_obs + start[k] * 12, *oa = R.opp_act + start[k] * 2;
            const int f = opp_frames(R, k);
            if (f > 1) {
                rc = R.tensor_cores ? ss_actor_forward_frames_tc(opp_prm(k), 0, 0, R.opp_stacks[k], f, head, oa, b, tiles, tile_bytes, stream)
                                    : ss_actor_forward_frames(opp_prm(k), 0, 0, (const float *)R.opp_stacks[k], f, head, oa, b, stream);
                ++k;
            } else if (R.tensor_cores) {
                int e = k + 1;                                // the run of 1-frame opponents [k, e): one launch
                while (e < K && opp_frames(R, e) == 1) ++e;
                rc = ss_actor_forward_segments_tc(opp_prm(k), R.opp_param_stride, seg_rows + k, e - k, oo, oa, stream);
                k = e;
            } else {
                rc = ss_actor_forward(opp_prm(k), oo, oa, b, 0.f, 1, 0.f, 0, 0, stream);
                ++k;
            }
        }
        if (rc != SS_OK) return rc;
        sslaunch::pdl_mode() = kOn;
        float *step_obs = F > 1 ? R.obs : ring ? R.ring_next_obs + seg * L * 12 : R.obs;
        rc = speeds ? ss_env_step_pool_speeds(R.state, n, M, (int)K, a, R.opp_act, step_obs, ring && F == 1 ? o_next : nullptr,
                                              ring ? R.ring_reward + seg * L : R.reward, ring ? R.ring_done + seg * L : nullptr,
                                              R.opp_obs, R.done, R.winner, R.reward_mode, R.tick_limit, R.reset_mode, R.env_seed,
                                              R.env_counter + (uint64_t)t, R.status, R.step_flags, R.pool_stats, R.opp_envs, R.speeds,
                                              stream)
           : R.opp_envs ? ss_env_step_pool_blocks(R.state, n, M, (int)K, a, R.opp_act, step_obs, ring && F == 1 ? o_next : nullptr,
                                                  ring ? R.ring_reward + seg * L : R.reward, ring ? R.ring_done + seg * L : nullptr,
                                                  R.opp_obs, R.done, R.winner, R.reward_mode, R.tick_limit, R.reset_mode, R.env_seed,
                                                  R.env_counter + (uint64_t)t, R.status, R.step_flags, R.pool_stats, R.opp_envs, stream)
                        : ss_env_step_pool(R.state, n, M, (int)K, a, R.opp_act, step_obs, ring && F == 1 ? o_next : nullptr,
                                           ring ? R.ring_reward + seg * L : R.reward, ring ? R.ring_done + seg * L : nullptr, R.opp_obs,
                                           R.done, R.winner, R.reward_mode, R.tick_limit, R.reset_mode, R.env_seed,
                                           R.env_counter + (uint64_t)t, R.status, R.step_flags, R.pool_stats, stream);
        if (rc != SS_OK) return rc;
        if (F > 1) {
            float *r1 = ring ? R.ring_next_obs + seg * L * w : R.rows, *r2 = !ring ? nullptr : !last ? R.ring_obs + nseg * L * w : R.rows;
            rc = ss_obs_stack_push_pool(R.tensor_cores ? R.stack_tc : nullptr, R.stack32, n, M, F, head + 1, R.obs, R.done, r1, r2, stream);
            if (rc != SS_OK) return rc;
        }
        for (int k = 0; k < K && M > 0 && rc == SS_OK; ++k) {
            const int f = opp_frames(R, k);
            if (f == 1) continue;
            const uint8_t *dk = R.done + S + start[k];
            float *oo = R.opp_obs + start[k] * 12;
            rc = R.tensor_cores ? ss_obs_stack_push_tc(R.opp_stacks[k], seg_rows[k], f, head + 1, oo, dk, 1, stream)
                                : ss_obs_stack_push((float *)R.opp_stacks[k], seg_rows[k], f, head + 1, oo, dk, 1, stream);
        }
        if (rc != SS_OK) return rc;
    }
    if (ring) {            // the last tick's actions and rewards for the caller's buffers
        seg = (seg + segs - 1) % segs;
        if (cudaMemcpyAsync(R.act, R.ring_act + seg * L * 2, (size_t)L * 8, cudaMemcpyDeviceToDevice, st) != cudaSuccess ||
            cudaMemcpyAsync(R.reward, R.ring_reward + seg * L, (size_t)L * 4, cudaMemcpyDeviceToDevice, st) != cudaSuccess)
            return SS_ERR_CUDA;
    }
    return SS_OK;
}

}  // namespace

extern "C" {

int64_t ss_pool_rollout_frames_workspace_bytes(const ss_pool_rollout_frames_args *args) { return args ? workspace_bytes(*args) : -1; }

int ss_pool_rollout_frames(const ss_pool_rollout_frames_args *args, void *stream) {
    return args ? rollout(*args, false, stream) : SS_ERR_INVALID_ARG;
}

int ss_pool_rollout_speeds(const ss_pool_rollout_frames_args *args, void *stream) {
    return args ? rollout(*args, true, stream) : SS_ERR_INVALID_ARG;
}

int ss_pool_rollout(const ss_pool_rollout_args *args, void *stream) {
    if (!args) return SS_ERR_INVALID_ARG;
    const ss_pool_rollout_args &P = *args;
    Args R = {};
    R.state = P.state; R.n_envs = P.n_envs; R.pool_envs = P.pool_envs; R.n_opponents = P.n_opponents;
    R.params = P.params; R.opp_params = P.opp_params; R.opp_param_stride = P.opp_param_stride;
    R.obs = P.obs; R.act = P.act; R.reward = P.reward; R.opp_obs = P.opp_obs; R.opp_act = P.opp_act;
    R.done = P.done; R.winner = P.winner;
    R.ring_obs = P.ring_obs; R.ring_act = P.ring_act; R.ring_reward = P.ring_reward; R.ring_next_obs = P.ring_next_obs;
    R.ring_done = P.ring_done; R.capacity = P.capacity; R.write_pos = P.write_pos; R.n_ticks = P.n_ticks;
    R.param_noise_sd = P.param_noise_sd; R.noise_group = P.noise_group; R.action_noise_sd = P.action_noise_sd;
    R.tensor_cores = P.tensor_cores; R.reward_mode = P.reward_mode; R.tick_limit = P.tick_limit; R.reset_mode = P.reset_mode;
    R.env_seed = P.env_seed; R.env_counter = P.env_counter; R.noise_seed = P.noise_seed; R.noise_counter = P.noise_counter;
    R.speeds = P.speeds; R.status = P.status; R.step_flags = P.step_flags; R.pool_stats = P.pool_stats;
    R.frames = 1;          // every network reads one frame: no history, no workspace
    return rollout(R, false, stream);
}

}  // extern "C"
