// ss_league.cu -- ss_league_play: n ticks of a league of up to SS_LEAGUE_MAX_POLICIES actors from one host call
// (include/skillshot_b200.h).
//
// A tick is the segments' forwards, one ss_env_step_seated and, for a segment whose policy reads a history of frames, the
// push of its newest observations.  Everything is an existing entry point; this file only decides which forward each
// segment takes and checks the arguments before anything is enqueued.  The observations are updated in place: the
// forwards read `obs` before the env step of the same tick overwrites it, in stream order.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/skillshot_b200.h"

namespace {

bool frames_ok(int f) { return f >= 1 && f <= SS_MAX_FRAMES; }

// the segment table and frame counts of L are usable: 2..SS_LEAGUE_MAX_POLICIES segments of >= 1 row each from row 0
bool segments_ok(const ss_league_args &L) {
    if (L.n_policies < 2 || L.n_policies > SS_LEAGUE_MAX_POLICIES || !L.seg_start || !L.frames || L.seg_start[0] != 0) return false;
    for (int s = 0; s < L.n_policies; ++s)
        if (L.seg_start[s + 1] <= L.seg_start[s] || !frames_ok(L.frames[s])) return false;
    return true;
}

}  // namespace

extern "C" {

// the frame-stacked tensor-core forward's scratch for the largest frames > 1 segment (the forwards run one after the other
// on one stream and share it)
int64_t ss_league_workspace_bytes(const ss_league_args *args) {
    if (!args || !segments_ok(*args)) return -1;
    if (!args->tensor_cores) return 0;
    int64_t need = 0;
    for (int s = 0; s < args->n_policies; ++s) {
        if (args->frames[s] == 1) continue;
        const int64_t b = ss_actor_frames_tc_workspace_bytes(args->seg_start[s + 1] - args->seg_start[s], 0);
        if (b > need) need = b;
    }
    return need;
}

int ss_league_play(const ss_league_args *args, void *stream) {
    if (!args) return SS_ERR_INVALID_ARG;
    const ss_league_args L = *args;
    const int64_t n = L.n_envs;
    if (!L.state || !L.seat_rows || !L.obs || !L.act || !L.params || n <= 0 || L.n_ticks <= 0 || L.head < 0 || L.tick_limit <= 0)
        return SS_ERR_INVALID_ARG;
    if (!segments_ok(L) || L.seg_start[L.n_policies] != 2 * n) return SS_ERR_INVALID_ARG;
    if (L.param_stride & 3) return SS_ERR_INVALID_ARG;
    for (int s = 0; s < L.n_policies; ++s) {
        if (L.param_stride < ss_actor_frames_params(L.frames[s])) return SS_ERR_INVALID_ARG;
        if (L.frames[s] > 1 && (!L.stacks || !L.stacks[s] || ((uintptr_t)L.stacks[s] & 15))) return SS_ERR_INVALID_ARG;
    }
    if ((((uintptr_t)L.state | (uintptr_t)L.obs | (uintptr_t)L.params | (uintptr_t)L.speeds | (uintptr_t)L.workspace) & 15) ||
        (((uintptr_t)L.act | (uintptr_t)L.seat_rows) & 7) || ((uintptr_t)L.status & 3))
        return SS_ERR_INVALID_ARG;
    const int64_t need = ss_league_workspace_bytes(&L);
    if (need > 0 && (!L.workspace || L.workspace_bytes < need)) return SS_ERR_INVALID_ARG;

    const int P = L.n_policies;
    int64_t rows[SS_LEAGUE_MAX_POLICIES];
    for (int s = 0; s < P; ++s) rows[s] = L.seg_start[s + 1] - L.seg_start[s];
    auto prm = [&](int s) { return L.params + s * L.param_stride; };
    auto obs = [&](int s) { return L.obs + L.seg_start[s] * SS_NUM_OBS; };
    auto act = [&](int s) { return L.act + L.seg_start[s] * SS_DIM_ACTION; };
    int64_t head = L.head;
    for (int t = 0; t < L.n_ticks; ++t) {
        int rc = SS_OK;
        for (int s = 0; s < P && rc == SS_OK;) {
            if (L.frames[s] > 1) {
                rc = L.tensor_cores ? ss_actor_forward_frames_tc(prm(s), 0, 0, L.stacks[s], L.frames[s], head, act(s), rows[s], L.workspace,
                                                                 L.workspace_bytes, stream)
                                    : ss_actor_forward_frames(prm(s), 0, 0, (const float *)L.stacks[s], L.frames[s], head, act(s),
                                                              rows[s], stream);
                ++s;
            } else if (L.tensor_cores) {
                int e = s + 1;                                // the run of frames-1 segments [s, e): one launch
                while (e < P && L.frames[e] == 1) ++e;
                rc = ss_actor_forward_segments_tc(prm(s), L.param_stride, rows + s, e - s, obs(s), act(s), stream);
                s = e;
            } else {
                rc = ss_actor_forward(prm(s), obs(s), act(s), rows[s], 0.f, 1, 0.f, 0, 0, stream);
                ++s;
            }
        }
        if (rc != SS_OK) return rc;
        rc = ss_env_step_seated(L.state, n, L.seat_rows, 2 * n, L.act, L.obs, L.tick_limit, L.speeds, L.status, stream);
        if (rc != SS_OK) return rc;
        ++head;
        for (int s = 0; s < P && rc == SS_OK; ++s) {
            if (L.frames[s] == 1) continue;
            // no auto-reset in a league: no history is ever refilled
            rc = L.tensor_cores ? ss_obs_stack_push_tc(L.stacks[s], rows[s], L.frames[s], head, obs(s), nullptr, 1, stream)
                                : ss_obs_stack_push((float *)L.stacks[s], rows[s], L.frames[s], head, obs(s), nullptr, 1, stream);
        }
        if (rc != SS_OK) return rc;
    }
    return SS_OK;
}

}  // extern "C"
