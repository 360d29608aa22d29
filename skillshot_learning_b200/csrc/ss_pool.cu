// ss_pool.cu -- ss_pool_rollout: n training ticks of the self-play learner with part of its envs played against a pool of
// frozen opponents, from one host call (include/skillshot_b200.h, "training against a pool").
//
// A tick is the learner's forward over its L rows, the opponents' segment forward over their M rows and ss_env_step_pool.
// Every kernel is an existing entry point; this file checks the arguments before anything is enqueued and lays the learner's
// rows into the replay ring as ss_selfplay_rollout does.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/skillshot_b200.h"
#include "ss_launch.cuh"

extern "C" {

int ss_pool_rollout(const ss_pool_rollout_args *args, void *stream) {
    if (!args) return SS_ERR_INVALID_ARG;
    const ss_pool_rollout_args R = *args;
    const int64_t n = R.n_envs, M = R.pool_envs, K = R.n_opponents;
    if (!R.state || !R.params || !R.obs || !R.act || !R.reward || !R.done || !R.winner || n <= 0 || R.n_ticks <= 0)
        return SS_ERR_INVALID_ARG;
    if (M < 0 || M > n) return SS_ERR_INVALID_ARG;
    if (M > 0) {
        if (K < 1 || K > SS_LEAGUE_MAX_POLICIES || M % (2 * K) != 0 || !R.opp_params || !R.opp_obs || !R.opp_act) return SS_ERR_INVALID_ARG;
        if ((R.opp_param_stride & 3) || R.opp_param_stride < 0 || (K > 1 && R.opp_param_stride < SS_ACTOR_PARAMS)) return SS_ERR_INVALID_ARG;
    }
    if (R.speeds) return SS_ERR_INVALID_ARG;
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
    const int64_t S = n - M, L = 2 * S + M, b = M > 0 ? M / K : 0;
    const bool ring = R.ring_obs != nullptr;
    // the transitions are produced in place (see ss_selfplay_rollout: one segment of L rows per tick, and with a single
    // segment the second observation copy would overwrite the rows the actor has just read)
    if (ring && (!R.ring_act || !R.ring_reward || !R.ring_next_obs || !R.ring_done || R.capacity <= 0 || R.capacity % L != 0 ||
                 R.write_pos < 0 || R.write_pos >= R.capacity || R.write_pos % L != 0 || (R.capacity / L < 2 && R.n_ticks != 1)))
        return SS_ERR_INVALID_ARG;

    cudaStream_t st = (cudaStream_t)stream;
    const int64_t segs = ring ? R.capacity / L : 1;
    int64_t seg = ring ? R.write_pos / L : 0;
    if (ring && cudaMemcpyAsync(R.ring_obs + seg * L * 12, R.obs, (size_t)L * 48, cudaMemcpyDeviceToDevice, st) != cudaSuccess)
        return SS_ERR_CUDA;
    int64_t seg_rows[SS_LEAGUE_MAX_POLICIES];
    for (int k = 0; k < K && M > 0; ++k) seg_rows[k] = b;
    // The launches of a tick form the dependent-launch chain of ss_selfplay_rollout (ss_launch.cuh).  The learner's forward
    // stages its parameters ahead of its wait from the second tick on (its predecessor, the env step, does not write them);
    // the opponents' forward always does (its predecessor, the learner's forward, does not write the opponents' vectors).
    const int kOn = (R.tensor_cores && sslaunch::chain_enabled()) ? sslaunch::kPdlOn : sslaunch::kPdlOff;
    sslaunch::PdlScope scope(kOn);
    const int kEarly = kOn ? (sslaunch::kPdlOn | sslaunch::kPdlEarlyWeights) : kOn;
    for (int t = 0; t < R.n_ticks; ++t, seg = (seg + 1) % segs) {
        float *o = ring ? R.ring_obs + seg * L * 12 : R.obs, *a = ring ? R.ring_act + seg * L * 2 : R.act;
        float *o_next = !ring ? R.obs : (t + 1 < R.n_ticks) ? R.ring_obs + ((seg + 1) % segs) * L * 12 : R.obs;
        sslaunch::pdl_mode() = t > 0 ? kEarly : kOn;
        const uint64_t nc = R.noise_counter + (uint64_t)t;
        int rc = R.tensor_cores ? ss_actor_forward_tc(R.params, o, a, L, R.param_noise_sd, R.noise_group, R.action_noise_sd, R.noise_seed,
                                                      nc, stream)
                                : ss_actor_forward(R.params, o, a, L, R.param_noise_sd, R.noise_group, R.action_noise_sd, R.noise_seed,
                                                   nc, stream);
        if (rc != SS_OK) return rc;
        if (M > 0) {
            sslaunch::pdl_mode() = kEarly;
            if (R.tensor_cores) {
                rc = ss_actor_forward_segments_tc(R.opp_params, R.opp_param_stride, seg_rows, (int)K, R.opp_obs, R.opp_act, stream);
            } else {
                for (int k = 0; k < K && rc == SS_OK; ++k)
                    rc = ss_actor_forward(R.opp_params + k * R.opp_param_stride, R.opp_obs + k * b * 12, R.opp_act + k * b * 2, b, 0.f, 1,
                                          0.f, 0, 0, stream);
            }
            if (rc != SS_OK) return rc;
        }
        sslaunch::pdl_mode() = kOn;
        rc = ss_env_step_pool(R.state, n, M, (int)K, a, R.opp_act, ring ? R.ring_next_obs + seg * L * 12 : R.obs, ring ? o_next : nullptr,
                              ring ? R.ring_reward + seg * L : R.reward, ring ? R.ring_done + seg * L : nullptr, R.opp_obs, R.done,
                              R.winner, R.reward_mode, R.tick_limit, R.reset_mode, R.env_seed, R.env_counter + (uint64_t)t, R.status,
                              R.step_flags, R.pool_stats, stream);
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

}  // extern "C"
