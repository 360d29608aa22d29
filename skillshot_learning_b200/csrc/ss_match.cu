// ss_match.cu -- ss_match_play: n ticks of a match between two actors from one host call (include/skillshot_b200.h).
//
// A tick is the policies' forwards, one ss_env_step_match and, for a policy that reads a history of frames, the push of its
// newest observation.  Everything is an existing entry point; this file only decides which forward each policy takes and
// checks the arguments before anything is enqueued.  The observations are updated in place: the forwards read `obs` before
// the env step of the same tick overwrites it, in stream order.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/skillshot_b200.h"

namespace {

// bytes of the frame-stacked tensor-core forward's scratch for one policy's n rows (shared by the two policies: their
// forwards run one after the other on the same stream)
int64_t frames_tc_bytes(int64_t n_envs, int frames) { return frames > 1 ? ss_actor_frames_tc_workspace_bytes(n_envs, 0) : 0; }

bool frames_ok(int f) { return f >= 1 && f <= SS_MAX_FRAMES; }

}  // namespace

extern "C" {

int64_t ss_match_workspace_bytes(int64_t n_envs, int frames_a, int frames_b, int tensor_cores) {
    if (n_envs <= 0 || !frames_ok(frames_a) || !frames_ok(frames_b)) return -1;
    if (!tensor_cores) return 0;
    const int64_t a = frames_tc_bytes(n_envs, frames_a), b = frames_tc_bytes(n_envs, frames_b);
    return a > b ? a : b;
}

int ss_match_play(const ss_match_args *args, void *stream) {
    if (!args) return SS_ERR_INVALID_ARG;
    const ss_match_args M = *args;
    const int64_t n = M.n_envs;
    if (!M.state || !M.obs || !M.act || !M.params || n <= 0 || M.n_ticks <= 0 || M.head < 0) return SS_ERR_INVALID_ARG;
    if (M.split < 0 || M.split > n || M.tick_limit <= 0) return SS_ERR_INVALID_ARG;
    if (!frames_ok(M.frames_a) || !frames_ok(M.frames_b)) return SS_ERR_INVALID_ARG;
    if ((M.frames_a > 1 && !M.stack_a) || (M.frames_b > 1 && !M.stack_b)) return SS_ERR_INVALID_ARG;
    const int64_t pa = ss_actor_frames_params(M.frames_a), pb = ss_actor_frames_params(M.frames_b);
    if (M.param_stride < (pa > pb ? pa : pb) || (M.param_stride & 3)) return SS_ERR_INVALID_ARG;
    if ((((uintptr_t)M.state | (uintptr_t)M.obs | (uintptr_t)M.params | (uintptr_t)M.speeds | (uintptr_t)M.stack_a |
          (uintptr_t)M.stack_b | (uintptr_t)M.workspace) & 15) ||
        ((uintptr_t)M.act & 7) || ((uintptr_t)M.status & 3))
        return SS_ERR_INVALID_ARG;
    const int64_t need = ss_match_workspace_bytes(n, M.frames_a, M.frames_b, M.tensor_cores);
    if (need > 0 && (!M.workspace || M.workspace_bytes < need)) return SS_ERR_INVALID_ARG;

    const float *params[2] = {M.params, M.params + M.param_stride};
    const int frames[2] = {M.frames_a, M.frames_b};
    void *stacks[2] = {M.stack_a, M.stack_b};
    float *obs[2] = {M.obs, M.obs + n * SS_NUM_OBS}, *act[2] = {M.act, M.act + n * SS_DIM_ACTION};
    const bool one_launch = M.tensor_cores && M.frames_a == 1 && M.frames_b == 1;
    int64_t head = M.head;
    for (int t = 0; t < M.n_ticks; ++t) {
        int rc = SS_OK;
        if (one_launch) {
            rc = ss_actor_forward_groups_tc(M.params, M.param_stride, n, M.obs, M.act, 2 * n, stream);
        } else {
            for (int p = 0; p < 2 && rc == SS_OK; ++p) {
                if (frames[p] > 1)
                    rc = M.tensor_cores ? ss_actor_forward_frames_tc(params[p], 0, 0, stacks[p], frames[p], head, act[p], n, M.workspace,
                                                                     M.workspace_bytes, stream)
                                        : ss_actor_forward_frames(params[p], 0, 0, (const float *)stacks[p], frames[p], head, act[p], n,
                                                                  stream);
                else
                    rc = M.tensor_cores ? ss_actor_forward_tc(params[p], obs[p], act[p], n, 0.f, 1, 0.f, 0, 0, stream)
                                        : ss_actor_forward(params[p], obs[p], act[p], n, 0.f, 1, 0.f, 0, 0, stream);
            }
        }
        if (rc != SS_OK) return rc;
        rc = ss_env_step_match(M.state, n, M.split, M.act, M.obs, M.tick_limit, M.speeds, M.status, stream);
        if (rc != SS_OK) return rc;
        ++head;
        for (int p = 0; p < 2 && rc == SS_OK; ++p) {
            if (frames[p] == 1) continue;
            // no auto-reset in a match: no history is ever refilled
            rc = M.tensor_cores ? ss_obs_stack_push_tc(stacks[p], n, frames[p], head, obs[p], nullptr, 1, stream)
                                : ss_obs_stack_push((float *)stacks[p], n, frames[p], head, obs[p], nullptr, 1, stream);
        }
        if (rc != SS_OK) return rc;
    }
    return SS_OK;
}

}  // extern "C"
