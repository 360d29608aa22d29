// ss_update.cu -- one DDPG update step enqueued by ONE host call.
//
// models_fit of the reference (SkillshotLearner.py:419-443) is, per minibatch, a critic fit
// step followed by model_actor_fit_step (386-417).  The batched build draws the minibatch from
// the device replay ring and may regress the critic on a TD target; every piece is its own
// entry point of this library (ss_replay_sample, ss_ddpg_targets*, ss_critic_grad*,
// ss_actor_grad*, ss_adam_tf, ss_peer_*).  Called one by one from Python they cost ~130-160 us
// of interpreter and ctypes time per update, about as much as the kernels themselves at a
// 65,536-row minibatch; this call issues the same launches, in the same order, with the same
// arguments, from C.  Nothing here touches the device directly.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/skillshot_b200.h"
#include "ss_launch.cuh"

#include <atomic>
#include <string.h>

int &sslaunch::pdl_mode() {
    static thread_local int mode = sslaunch::kPdlOff;
    return mode;
}

static std::atomic<int> g_chain_override{-1};       // -1: the default (chained)

bool sslaunch::chain_enabled() { return g_chain_override.load(std::memory_order_relaxed) != 0; }

extern "C" int ss_set_dependent_launch(int enabled) {
    return g_chain_override.exchange(enabled < 0 ? -1 : (enabled ? 1 : 0), std::memory_order_relaxed);
}

extern "C" int ss_ddpg_update(const ss_ddpg_update_args *a, void *stream) {
    if (!a || !a->ring_obs || !a->ring_act || !a->ring_reward || !a->ring_next_obs || !a->ring_done || a->batch < 1 ||
        a->size < 1 || a->size > a->capacity || !a->obs || !a->act || !a->reward || !a->next_obs || !a->done || !a->actor ||
        !a->critic || !a->m_actor || !a->v_actor || !a->m_critic || !a->v_critic || !a->stats || !a->workspace ||
        a->step_actor < 1 || a->step_critic < 1)
        return SS_ERR_INVALID_ARG;
    const bool peers = a->peer_bases != nullptr;
    if (peers && (a->world < 1 || a->world > SS_PEER_MAX_WORLD || a->rank < 0 || a->rank >= a->world || a->epoch == 0 ||
                  !a->done_counter))
        return SS_ERR_INVALID_ARG;
    if (a->gamma != 0.f && (!a->y || !a->target_actor || !a->target_critic)) return SS_ERR_INVALID_ARG;
    if (a->n_step < 0 || a->n_step > SS_REPLAY_MAX_NSTEP) return SS_ERR_INVALID_ARG;
    const int64_t n = a->batch;
    const bool tc = a->tensor_cores != 0;
    int rc;
    // Single GPU: the launches of this call form one dependent chain (ss_launch.cuh): each grid's CTAs are placed while its
    // predecessor drains and hold at griddepcontrol.wait.  kEarly additionally lets a tensor-core kernel stage its network's
    // parameters ahead of that wait; it is given to exactly the launches whose immediate predecessor does not write those
    // parameters (the one before that is complete by then, see the header):
    //   sample -> [actor'(s2) -> critic'(s2, a2)] -> critic gradient     none of the predecessors writes parameters
    //   reduce + Adam (critic, critic') -> actor(s)                        reads the actor
    //   actor(s) -> critic(s, a)                                           Adam is two launches back
    //     (as ONE pair launch the critic role directly follows Adam and stages behind its wait: kPdlPairCriticLate)
    //   critic(s, a) -> actor gradient -> reduce + Adam (actor, actor')
    // With the peer exchange the order is ... critic gradient -> push -> actor(s) -> peers' Adam (critic) -> critic(s, a) -> ...:
    // critic(s, a) then directly follows the kernel that writes the critic and stages behind its wait (kPdlEarlyAfterFirst).
    // ss_set_dependent_launch(0) switches the chain off (the equality test).
    const int kOn = sslaunch::chain_enabled() ? sslaunch::kPdlOn : sslaunch::kPdlOff;
    const int kEarly = kOn ? (sslaunch::kPdlOn | sslaunch::kPdlEarlyWeights) : sslaunch::kPdlOff;
    sslaunch::PdlScope scope(kOn);

    // minibatch (uniform with replacement from the filled part of the ring); drawn beside the previous launch's tail when the
    // caller vouches for it (args.sample_early)
    if (kOn && a->sample_early) sslaunch::pdl_mode() = kOn | sslaunch::kPdlSampleEarly;
    // (n-step rows: the same draw over the eligible runs, then the walk; a->gamma is g_n)
    if (a->n_step > 1)
        rc = ss_replay_sample_nstep(a->ring_obs, a->ring_act, a->ring_reward, a->ring_next_obs, a->ring_done, a->capacity, 1,
                                    a->tick_rows, a->n_step, a->step_gamma, a->runs_host, a->n_runs, a->replay_seed,
                                    a->replay_counter, n, a->obs, a->act, a->reward, a->next_obs, a->done, a->indices, nullptr,
                                    stream);
    else
        rc = ss_replay_sample(a->ring_obs, a->ring_act, a->ring_reward, a->ring_next_obs, a->ring_done, a->capacity, a->size,
                              nullptr, a->replay_seed, a->replay_counter, n, a->obs, a->act, a->reward, a->next_obs, a->done,
                              a->indices, stream);
    if (rc != SS_OK) return rc;

    // critic target: the reference regresses on the reward itself (gamma = 0, SkillshotLearner.py:434)
    const float *y = a->reward;
    sslaunch::pdl_mode() = kEarly;
    if (a->gamma != 0.f) {
        rc = tc ? ss_ddpg_targets_tc_paired(a->target_actor, a->target_critic, a->reward, a->next_obs, a->done, a->gamma, a->y, n,
                                            a->workspace, a->workspace_bytes, a->pair_mail, stream)
                : ss_ddpg_targets(a->target_actor, a->target_critic, a->reward, a->next_obs, a->done, a->gamma, a->y, n, stream);
        if (rc != SS_OK) return rc;
        y = a->y;
    }

    // critic: gradient of the batch-mean squared error -> (exchange) -> Adam (+ soft target update).  The gradient
    // kernels leave per-CTA slices; one more kernel sums them in a fixed order and applies Adam (ss_reduce_adam_tf), or
    // pushes the sum to every rank's inbox (ss_peer_reduce_push) for the peers' Adam kernel.
    auto critic_grad = tc ? ss_critic_grad_tc : ss_critic_grad;
    rc = critic_grad(a->critic, a->obs, a->act, y, nullptr, a->dropout_rate, a->seed, a->counter, n, a->n_global, a->row_offset,
                     nullptr, a->stats, a->workspace, a->workspace_bytes, stream);
    if (rc <= 0) return rc < 0 ? rc : SS_ERR_INVALID_ARG;
    sslaunch::pdl_mode() = kOn;
    // The actor step begins with a = actor(s), which needs neither the critic's new weights nor anything the exchange
    // delivers: on the tensor-core path of a sharded update it is enqueued BETWEEN the push of this rank's critic gradient and
    // the Adam kernel that waits for the peers' pushes, so that the exchange's latency (rank skew + NVLink visibility,
    // ~20 us on 8 GPUs) passes under 15 us of useful work instead of an idle spin.  (The gradient slices of the critic step
    // have been consumed by the push kernel by then; the actions land in the scratch area behind the slices.)
    // Push, wait and Adam as ONE kernel per exchange (ss_peer_reduce_adam_tf) is bit-identical and was measured SLOWER:
    // 0.203 vs 0.189 ms per update on 2 GPUs (profiles/r2_peer_fused_ab_n2.txt) -- 573 CTAs each fencing and polling at
    // system scope cost more than the kernel boundary they remove, and nothing runs under the wait any more.
    const bool early_actor_forward = peers && tc;
    if (peers) {
        rc = ss_peer_reduce_push(a->workspace, rc, SS_CRITIC_PARAMS, a->stats, a->peer_bases, a->world, a->rank,
                                 a->peer_capacity, a->epoch, a->done_counter, stream);
        if (rc != SS_OK) return rc;
        if (early_actor_forward) {
            sslaunch::pdl_mode() = kEarly;
            rc = ss_actor_grad_tc_staged(a->actor, a->critic, a->obs, n, nullptr, a->stats + 1, a->workspace, a->workspace_bytes, 1,
                                         stream);
            if (rc != SS_OK) return rc;
            sslaunch::pdl_mode() = kOn;
        }
        rc = ss_peer_adam_tf(a->peer_bases[a->rank], a->world, a->peer_capacity, a->epoch, a->critic, a->m_critic, a->v_critic,
                             a->target_critic, a->grad_critic, SS_CRITIC_PARAMS, a->step_critic, a->lr_critic, a->beta1,
                             a->beta2, a->eps, a->tau, 1.0f, a->status, stream);
    } else {
        rc = ss_reduce_adam_tf(a->workspace, rc, SS_CRITIC_PARAMS, a->stats, a->grad_critic, a->critic, a->m_critic, a->v_critic,
                               a->target_critic, a->step_critic, a->lr_critic, a->beta1, a->beta2, a->eps, a->tau, 1.0f, stream);
    }
    if (rc != SS_OK) return rc;

    // actor: model_actor_fit_step with the critic just updated (SkillshotLearner.py:440-443 follows 434)
    sslaunch::pdl_mode() = kEarly;
    if (early_actor_forward && kOn) sslaunch::pdl_mode() = kOn | sslaunch::kPdlEarlyAfterFirst;
    else if (kOn && tc && a->pair_mail) sslaunch::pdl_mode() = kEarly | sslaunch::kPdlPairCriticLate;   // the pair follows Adam(critic)
    if (early_actor_forward)
        rc = ss_actor_grad_tc_staged(a->actor, a->critic, a->obs, n, nullptr, a->stats + 1, a->workspace, a->workspace_bytes, 2, stream);
    else if (tc)
        rc = ss_actor_grad_tc_paired(a->actor, a->critic, a->obs, n, nullptr, a->stats + 1, a->workspace, a->workspace_bytes, 0,
                                     a->pair_mail, stream);
    else
        rc = ss_actor_grad(a->actor, a->critic, a->obs, n, nullptr, a->stats + 1, a->workspace, a->workspace_bytes, stream);
    if (rc <= 0) return rc < 0 ? rc : SS_ERR_INVALID_ARG;
    sslaunch::pdl_mode() = kOn;
    if (peers) {
        rc = ss_peer_reduce_push(a->workspace, rc, SS_ACTOR_PARAMS, a->stats + 1, a->peer_bases, a->world, a->rank,
                                 a->peer_capacity, a->epoch + 1, a->done_counter, stream);
        if (rc != SS_OK) return rc;
        rc = ss_peer_adam_tf(a->peer_bases[a->rank], a->world, a->peer_capacity, a->epoch + 1, a->actor, a->m_actor, a->v_actor,
                             a->target_actor, a->grad_actor, SS_ACTOR_PARAMS, a->step_actor, a->lr_actor, a->beta1, a->beta2,
                             a->eps, a->tau, 1.0f, a->status, stream);
    } else {
        rc = ss_reduce_adam_tf(a->workspace, rc, SS_ACTOR_PARAMS, a->stats + 1, a->grad_actor, a->actor, a->m_actor, a->v_actor,
                               a->target_actor, a->step_actor, a->lr_actor, a->beta1, a->beta2, a->eps, a->tau, 1.0f, stream);
    }
    return rc;
}
